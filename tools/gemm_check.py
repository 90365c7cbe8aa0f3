import os, sys, ctypes as C, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge; ge.build()
from fpv_drone_rl_agent_b200 import _lib
L = C.CDLL(_lib.LIB_PATH)
L.ppo_test_gemm.restype = C.c_int
L.ppo_test_gemm.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
torch.manual_seed(0)
for (n, k) in [(16, 16), (32, 32), (128, 128), (256, 32), (16, 256), (64, 64)]:
    A = torch.randn(128, k, device="cuda").to(torch.bfloat16)
    B = torch.randn(n, k, device="cuda").to(torch.bfloat16)
    D = torch.zeros(128, n, device="cuda")
    rc = L.ppo_test_gemm(A.data_ptr(), B.data_ptr(), D.data_ptr(), n, k, None)
    torch.cuda.synchronize()
    ref = A.float() @ B.float().t()
    err = (D - ref).abs().max().item()
    print(f"n={n} k={k} rc={rc} max_err={err:.3e} ref_max={ref.abs().max().item():.2f}", "OK" if err < 1e-2 * max(1.0, ref.abs().max().item()) else "MISMATCH")
    if err > 1: 
        print(D[:4,:8]); print(ref[:4,:8])
