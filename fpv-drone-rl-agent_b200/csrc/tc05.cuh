// tc05.cuh -- minimal hand-written wrappers of the sm_100a tensor-core path:
// tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM), TMEM alloc / ld,
// shared-memory matrix descriptors and the mbarrier the MMA commits to.
//
// Operand layout used everywhere in this repo: K-major, no swizzle
// ("interleaved"), stored as [K/8][rows][8] bf16 -- a core matrix is 8 rows x
// 16 bytes = 128 contiguous bytes; successive 8-row groups are SBO = 128 B
// apart, successive 8-column K chunks are LBO = rows * 16 B apart.  One
// tcgen05.mma consumes K = 16 (two K chunks); the next K step starts 2 * LBO
// further.  A weight matrix W[out][in] (PyTorch Linear layout) is exactly a
// K-major B operand with rows = out.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tc05 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- shared-memory matrix descriptor (SM100 UMMA SmemDescriptor) ----------
//  [0,14)  start address >> 4      [16,30) leading-dim byte offset >> 4 (K chunks)
//  [32,46) stride-dim byte offset >> 4 (8-row groups)   [46,48) version = 1
//  [49,52) base offset = 0   [52] lbo mode = 0   [61,64) layout = 0 (no swizzle)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// ---- instruction descriptor, kind::f16: D = fp32, A = B = bf16, both K-major
__host__ __device__ constexpr uint32_t make_idesc_bf16(uint32_t m, uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}

// all previously issued MMAs of this thread arrive on the mbarrier when done
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (tensor core reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM -------------------------------------------------------------------
// one full warp; ncols power of two >= 32; base address lands in *slot (smem)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(ncols) : "memory");
}

// thread t of warp w reads lane 32*(w%4)+t, 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- mbarrier -----------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// ---- operand staging helpers ------------------------------------------------------
// byte offset of the 16-byte chunk holding elements (row, 8*kc .. 8*kc+7)
__device__ __forceinline__ uint32_t chunk_off(uint32_t row, uint32_t kc, uint32_t rows) { return kc * rows * 16u + row * 16u; }

// W[rows][K] bf16 row-major in global -> interleaved K-major in smem; all threads of the CTA
__device__ __forceinline__ void stage_weight(uint8_t* smem, const __nv_bfloat16* __restrict__ w, uint32_t rows, uint32_t K,
                                             uint32_t tid, uint32_t nthreads) {
  const uint32_t kcs = K >> 3;
  for (uint32_t idx = tid; idx < rows * kcs; idx += nthreads) {
    const uint32_t r = idx / kcs, kc = idx - r * kcs;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(w + (size_t)r * K + kc * 8));
    *reinterpret_cast<uint4*>(smem + chunk_off(r, kc, rows)) = v;
  }
}

// ---- the slot scheme of the persistent MLP kernels -----------------------------------------------------------------
// A CTA runs several independent "slots" (groups of consecutive warps), each walking its own sequence of 128-row tiles, so
// that one slot's epilogue overlaps another slot's tcgen05.mma chain.  A slot synchronises on its own named barrier
// (id slot + 1; id 0 is __syncthreads).
__device__ __forceinline__ void slot_barrier(int slot, uint32_t slot_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "r"(slot_threads) : "memory");
}

// Slot-major tile order: tile t belongs to CTA t % grid, so the tiles that do not fill a whole round of grid x slots are
// spread over the CTAs instead of giving the first CTAs a tile in every slot.  Slot `slot` of CTA `cta` starts at the
// returned tile and steps by grid * slots.
__device__ __forceinline__ int slot_major_first_tile(int slot, int cta, int grid) { return slot * grid + cta; }

// Row `src[0 .. cols)` of an fp32 matrix -> x[0 .. cols), zeros beyond.  vec: src is 16-byte aligned (base pointer and row
// stride decided once per launch on the host, so the branch is uniform): float4 loads where four columns fit, scalar ones
// elsewhere.
template <int N>
__device__ __forceinline__ void load_f32_row(const float* __restrict__ src, int cols, bool vec, float (&x)[N]) {
  static_assert(N % 4 == 0, "whole float4 groups");
#pragma unroll
  for (int j = 0; j < N; ++j) x[j] = 0.f;
  if (vec) {
#pragma unroll
    for (int v = 0; v < N / 4; ++v)
      if (4 * v + 4 <= cols) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(src + 4 * v));
        x[4 * v] = t.x; x[4 * v + 1] = t.y; x[4 * v + 2] = t.z; x[4 * v + 3] = t.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (4 * v + j < cols) x[4 * v + j] = __ldg(src + 4 * v + j);
      }
  } else {
#pragma unroll
    for (int j = 0; j < N; ++j)
      if (j < cols) x[j] = __ldg(src + j);
  }
}

}  // namespace tc05
