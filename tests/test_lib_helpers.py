"""CPU: the argument check and the device normalisation that the Python bindings put in front of every library call
(_lib.expect, _lib.cuda_device).  A buffer the kernels would address wrongly must be refused with the argument's name."""
import pytest
import torch

from fpv_drone_rl_agent_b200 import _lib

CPU = torch.device("cpu")


def test_expect_accepts_matching_tensors():
    x = torch.zeros(4, 3)
    _lib.expect(x, "x", dtype=torch.float32, device=CPU)
    _lib.expect(x, "x", dtype=torch.float32, device=CPU, shape=(4, 3))
    _lib.expect(x, "x", dtype=torch.float32, device=CPU, shape=[4, 3], numel=12)
    _lib.expect(torch.zeros(6, 8)[2:6], "x", dtype=torch.float32, device=CPU, numel=32)  # a row slice is contiguous
    _lib.expect(x.bfloat16(), "x", dtype=(torch.float32, torch.bfloat16), device=CPU, shape=(4, 3))


@pytest.mark.parametrize("t, kw", [
    (torch.zeros(4, 3, dtype=torch.float64), {}),  # dtype
    (torch.zeros(4, 3, dtype=torch.uint8), dict(dtype=(torch.float32, torch.bfloat16))),  # none of several dtypes
    (torch.zeros(4, 3), dict(device=torch.device("cuda", 0))),  # device
    (torch.zeros(3, 4).t(), {}),  # transposed
    (torch.zeros(4, 6)[:, :3], {}),  # column view
    (torch.zeros(8, 3)[::2], {}),  # row step
    (torch.zeros(4, 4), dict(shape=(4, 3))),  # shape
    (torch.zeros(12), dict(shape=(4, 3))),  # the right number of elements in another shape
    (torch.zeros(4, 4), dict(numel=12)),  # numel
    (torch.zeros(4, 3), dict(shape=(4, 3), numel=13)),  # shape right, numel wrong
])
def test_expect_rejects_with_the_argument_name(t, kw):
    kw = dict(dict(dtype=torch.float32, device=CPU), **kw)
    with pytest.raises(ValueError, match=r"^obs_norm: expected a contiguous "):
        _lib.expect(t, "obs_norm", **kw)


def test_cuda_device_carries_an_index(monkeypatch):
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 5)
    assert _lib.cuda_device(None) == torch.device("cuda", 5)
    assert _lib.cuda_device("cuda") == torch.device("cuda", 5)
    assert _lib.cuda_device(torch.device("cuda")) == torch.device("cuda", 5)
    assert _lib.cuda_device("cuda:1") == torch.device("cuda", 1)
    assert _lib.cuda_device(torch.device("cuda", 2)) == torch.device("cuda", 2)
    assert _lib.cuda_device(3) == torch.device("cuda", 3)
    assert _lib.cuda_device(0) == torch.device("cuda", 0)


@pytest.mark.parametrize("device", ["cpu", torch.device("cpu"), "meta"])
def test_cuda_device_rejects_other_devices(device):
    with pytest.raises(ValueError, match="CUDA device"):
        _lib.cuda_device(device)
