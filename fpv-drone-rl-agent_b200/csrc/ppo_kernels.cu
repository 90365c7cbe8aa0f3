// ppo_kernels.cu -- on-device PPO rollout kernels for sm_100a (C-ABI: include/ppo_b200.h).
//   K2  actor-critic MLP forward on tcgen05 tensor cores + Gaussian sampling + log-prob
//   K3  GAE / returns reverse scan
//   K4  VecNormalize running statistics (obs and discounted-return) + reward normalisation
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>

#include "../../include/ppo_b200.h"
#include "../../include/quadx_b200.h"
#include "qx_internal.h"
#include "qx_model.cuh"
#include "tc05.cuh"

namespace ppo {

using namespace tc05;

// ---------------------------------------------------------------------------
// test hook: one 128 x n x k GEMM through the same staging / descriptor / TMEM
// helpers the policy kernel uses
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128) test_gemm_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ B,
                                                        float* __restrict__ D, int n, int k) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_slot;
  uint8_t* sA = smem;
  uint8_t* sB = smem + 128 * k * 2;
  const uint32_t tid = threadIdx.x, warp = tid >> 5;
  stage_weight(sA, A, 128, k, tid, 128);
  stage_weight(sB, B, n, k, tid, 128);
  fence_async_smem();
  uint32_t ncols = 32;
  while ((int)ncols < n) ncols <<= 1;
  if (warp == 0) tmem_alloc(&tmem_slot, ncols);
  if (tid == 0) { mbar_init(&bar, 1); mbar_fence_init(); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tbase = tmem_slot;
  if (tid == 0) {
    const uint32_t idesc = make_idesc_bf16(128, n);
    const uint32_t lboA = 128 * 16, lboB = n * 16;
    for (int ks = 0; ks < k / 16; ++ks)
      mma_bf16(tbase, make_desc(smem_u32(sA) + ks * 2 * lboA, lboA, 128), make_desc(smem_u32(sB) + ks * 2 * lboB, lboB, 128), idesc, ks > 0);
    mma_commit(&bar);
  }
  mbar_wait(&bar, 0);
  fence_after_sync();
  for (int c0 = 0; c0 < n; c0 += 16) {
    uint32_t r[16];
    tmem_ld16(tbase + ((warp * 32u) << 16) + c0, r);
    tmem_ld_wait();
    for (int j = 0; j < 16; ++j) D[(size_t)tid * n + c0 + j] = __uint_as_float(r[j]);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tbase, ncols);
}


// ---------------------------------------------------------------------------
// K2: ActorCriticPolicy.forward.  Persistent CTAs, one per SM, 768 threads = three
// independent "slots" of 256 threads; each slot walks its own sequence of
// 128-row tiles, so while one slot waits for its tcgen05.mma chain the others
// run their bias + tanh epilogues (tensor pipe, TMEM reads and the MUFU pipe
// overlap across slots).  All weights stay resident in
// shared memory in the interleaved K-major layout; per tile and slot
//   [L1p]      X[128x32]    . W1p^T          -> acc (TMEM 128 cols)
//   [L2p]      H1p[128x128] . W2p^T          -> acc
//   [L3p, L1v] H2p . W3p^T -> out (16 cols: action means);  X . W1v^T -> acc
//   [L2v]      H1v . W2v^T                   -> acc
//   [L3v]      H2v . W3v^T  accumulated into out (column act_dim: value)
// Each [..] is one commit -> mbarrier wait; after it the slot's 8 warps read
// the accumulator with tcgen05.ld 32x32b (warp w: TMEM lanes 32 (w % 4).., 64
// columns (w / 4)), add the bias, tanh, pack to bf16 and store the next A
// operand.  thread == accumulator row in the final epilogue (sampling).
// ---------------------------------------------------------------------------
constexpr int kHid = PPO_HIDDEN, kIn = PPO_IN_PAD, kHead = PPO_HEAD_PAD;
#ifndef PPO_SLOTS
#define PPO_SLOTS 3
#endif
constexpr int kSlots = PPO_SLOTS, kSlotThreads = 256, kFwdThreads = kSlots * kSlotThreads;
constexpr uint32_t kSmW1 = 0;                                  // [4][256][16 B]   rows 0..127 pi, 128..255 vf
constexpr uint32_t kSmW2p = kSmW1 + 2 * kHid * kIn * 2;        // [16][128][16 B]
constexpr uint32_t kSmW2v = kSmW2p + kHid * kHid * 2;
constexpr uint32_t kSmW3 = kSmW2v + kHid * kHid * 2;           // [32][16][16 B]   K chunks 0..15 pi half, 16..31 vf half
constexpr uint32_t kSmSlot = kSmW3 + kHead * 2 * kHid * 2;     // per slot: X [4][128][16 B] then H [16][128][16 B]
constexpr uint32_t kSlotX = 0, kSlotH = 128 * kIn * 2, kSlotBytes = kSlotH + 128 * kHid * 2;
constexpr uint32_t kSmB1 = kSmSlot + kSlots * kSlotBytes;      // 256 f32
constexpr uint32_t kSmB2 = kSmB1 + 2 * kHid * 4;
constexpr uint32_t kSmB3 = kSmB2 + 2 * kHid * 4;               // 16 f32
constexpr uint32_t kSmNorm = kSmB3 + kHead * 4;                // mean[32], inv_std[32]
constexpr uint32_t kSmTotal = kSmNorm + 2 * kIn * 4;
constexpr uint32_t kTmemCols = 512, kSlotTmem = 160, kTmemOut = 128;  // per slot: acc cols [0,128), out cols [128,144)
static_assert(kSlots * kSlotTmem <= kTmemCols && kSmTotal <= 227 * 1024, "slots must fit TMEM and shared memory");

struct FwdArgs {
  PpoPolicy p;
  const float* obs;
  int64_t obs_stride, n;
  const float* obs_mean;
  const float* obs_inv_std;
  float obs_clip;
  uint32_t seed_lo, seed_hi;
  uint64_t row0, step;
  int32_t deterministic;
  float* actions;
  float* env_actions;
  float* values;
  float* log_probs;
  float* obs_norm_out;            // [n, obs_dim] normalised obs as the policy saw them (what PPO stores)
  const uint64_t* step_base;      // device counter added to `step` (CUDA-graph replays)
  // gather / bootstrap mode: rows are taken from idx[0 .. *count) and, for rows that were truncated but not
  // terminated, reward[row] += gamma * V(obs[row])   (SB3 collect_rollouts time-limit bootstrap)
  const uint32_t* gather_idx;
  const uint32_t* gather_count;
  float* boot_reward;
  const uint8_t* boot_te;
  const uint8_t* boot_tr;
  float boot_gamma;
  int32_t grid;                   // CTAs of this launch (= gridDim.x), as a parameter so that the tile walk needs no register for it
  // fused VecNormalize update (ppo_policy_forward_stats): the launch first merges the raw rows of `obs` into the running
  // statistics {mean, var, count} (fp64) and refreshes the fp32 (mean, inv_std) it then normalises with -- see the kernel
  double* fs_stats;               // null = off (obs_mean / obs_inv_std are read as given)
  double* fs_scratch;             // per-CTA partial sums + ticket / flag words (ppo_running_stats_scratch_bytes)
  float fs_eps;
  float* fs_mean_out;             // == obs_mean, writable
  float* fs_inv_out;              // == obs_inv_std, writable
  int32_t pdl_wait;               // launched as a programmatic dependent of the statistics kernel: wait for it before reading its results
  int32_t boot_store;             // bootstrap: reward[row] = gamma V (the reward-normalisation launch that follows adds its result) instead of +=
  // 16-byte vector paths, decided on the host (fwd_vector_flags) so that the branches are uniform: a column slice of a wider
  // buffer, or a tensor at an odd storage offset, has a base pointer that is not 16-byte aligned and takes the scalar paths
  int32_t obs_vec;                // obs rows as float4: obs 16-byte aligned and obs_stride % 4 == 0
  int32_t norm_vec;               // obs_norm_out rows as float4: obs_norm_out 16-byte aligned and obs_dim % 4 == 0
  int32_t act_vec;                // actions / env_actions rows as float4: act_dim == 4 and both (where given) 16-byte aligned
};

// (defined with the K4 kernels below)
constexpr int kStatMaxDim = 32;
__device__ __forceinline__ bool last_block_done(unsigned int* ticket);
__device__ __forceinline__ void welford_merge_block(const double* part, int nblocks, int64_t n, int dim, double* __restrict__ stats, float eps,
                                                    float* __restrict__ mean_f32, float* __restrict__ inv_std_f32);
__device__ __forceinline__ unsigned int* stat_words(double* scratch);

__device__ __forceinline__ uint32_t tanh_pack_bf16x2(float lo, float hi) {
#ifdef PPO_TANH_BF16X2
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  uint32_t u = *reinterpret_cast<uint32_t*>(&v), r;
  asm("tanh.approx.bf16x2 %0, %1;" : "=r"(r) : "r"(u));
  return r;
#else
  float a, b;
  asm("tanh.approx.f32 %0, %1;" : "=f"(a) : "f"(lo));
  asm("tanh.approx.f32 %0, %1;" : "=f"(b) : "f"(hi));
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
#endif
}

// test hook: the hidden epilogue's activation on its own -- out[2i], out[2i + 1] = tanh_pack_bf16x2(x[2i], x[2i + 1]) (lo, hi)
__global__ void __launch_bounds__(256) test_tanh_kernel(const float* __restrict__ x, uint16_t* __restrict__ out, int64_t n) {
  const int64_t i = 2 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
  if (i >= n) return;
  const uint32_t r = tanh_pack_bf16x2(x[i], i + 1 < n ? x[i + 1] : 0.f);
  out[i] = (uint16_t)(r & 0xffffu);
  if (i + 1 < n) out[i + 1] = (uint16_t)(r >> 16);
}

// optional phase-timing buffer (debug / tuning only, see tools/k2_phases.py): [tile iteration][16] clock64 stamps of CTA 0, slot 0
__device__ long long* g_phase_clk = nullptr;
#define PHASE_STAMP(k) do { if (dbg && st == 0 && it < 8) dbg[it * 16 + (k)] = clock64(); } while (0)

__device__ __forceinline__ void slot_sync(int slot) { asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "r"(kSlotThreads) : "memory"); }

// bias + tanh + bf16 of this warp's 64 accumulator columns of this thread's row -> H chunks (A operand of the next layer)
__device__ __forceinline__ void hidden_epilogue(uint32_t tacc, const float* __restrict__ bias, uint8_t* sH, uint32_t row, int col0) {
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int c0 = col0 + 32 * half;
    uint32_t r[32];
    tmem_ld32(tacc + c0, r);
    tmem_ld_wait();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint4 v;
      const float4 b0 = *reinterpret_cast<const float4*>(bias + c0 + 8 * q), b1 = *reinterpret_cast<const float4*>(bias + c0 + 8 * q + 4);
      v.x = tanh_pack_bf16x2(__uint_as_float(r[8 * q + 0]) + b0.x, __uint_as_float(r[8 * q + 1]) + b0.y);
      v.y = tanh_pack_bf16x2(__uint_as_float(r[8 * q + 2]) + b0.z, __uint_as_float(r[8 * q + 3]) + b0.w);
      v.z = tanh_pack_bf16x2(__uint_as_float(r[8 * q + 4]) + b1.x, __uint_as_float(r[8 * q + 5]) + b1.y);
      v.w = tanh_pack_bf16x2(__uint_as_float(r[8 * q + 6]) + b1.z, __uint_as_float(r[8 * q + 7]) + b1.w);
      *reinterpret_cast<uint4*>(sH + chunk_off(row, (uint32_t)(c0 >> 3) + q, 128)) = v;
    }
  }
}

// raw observation columns [16 xh, 16 xh + 16) of row `xrow` of `tile` -> x[16] (zeros beyond obs_dim / n_rows)
__device__ __forceinline__ void load_obs_chunks(const FwdArgs& a, int64_t tile, int64_t n_rows, uint32_t xrow, uint32_t xh, int obs_dim, float (&x)[16]) {
#pragma unroll
  for (int j = 0; j < 16; ++j) x[j] = 0.f;
  if (tile * 128 + xrow >= n_rows) return;
  const int64_t xr = a.gather_idx ? (int64_t)a.gather_idx[tile * 128 + xrow] : tile * 128 + xrow;
  const float* src = a.obs + xr * a.obs_stride + 16 * xh;
  const int c0 = 16 * (int)xh;
  if (a.obs_vec) {
#pragma unroll
    for (int v = 0; v < 4; ++v)
      if (c0 + 4 * v + 4 <= obs_dim) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(src + 4 * v));
        x[4 * v] = t.x; x[4 * v + 1] = t.y; x[4 * v + 2] = t.z; x[4 * v + 3] = t.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (c0 + 4 * v + j < obs_dim) x[4 * v + j] = __ldg(src + 4 * v + j);
      }
  } else {
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (c0 + j < obs_dim) x[j] = __ldg(src + j);
  }
}

__global__ void __launch_bounds__(kFwdThreads, 1) policy_forward_kernel(const FwdArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bars[kSlots];
  __shared__ uint32_t tmem_slot;
  const uint32_t tid = threadIdx.x;
  const int slot = tid / kSlotThreads;
  const uint32_t st = tid % kSlotThreads, swarp = st >> 5, lane = tid & 31;   // thread / warp within the slot
  const uint32_t erow = (swarp & 3) * 32 + lane;   // accumulator row this thread reads in the epilogues
  const int ecol0 = (int)(swarp >> 2) * 64;        // and its 64 columns
  const uint32_t xrow = st & 127, xh = st >> 7;    // X-tile staging: row, pair of 8-column chunks
  const int obs_dim = a.p.obs_dim, act_dim = a.p.act_dim;
#ifdef PPO_K2_TRACE  // tuning builds only (QX_NVCC_EXTRA=-DPPO_K2_TRACE, tools/k2_phases.py): kernel entry / prologue / exit stamps of CTA 0
#define K2_TRACE(slot_) do { if (g_phase_clk && blockIdx.x == 0 && tid == 0) g_phase_clk[slot_] = clock64(); } while (0)
#else
#define K2_TRACE(slot_) do { } while (0)
#endif
  K2_TRACE(127);
  // gather mode (time-limit bootstrap): most steps have no truncated env at all -- leave before staging 88 KB of weights
  if (a.gather_idx && (int64_t)blockIdx.x * 128 >= (int64_t)*a.gather_count) return;  // (slot-major tile order: this CTA's first tile is blockIdx.x)
  // ---- fused VecNormalize update, first half: this CTA's share of the rows -> fp64 column sums (lane = column, the 24 warps
  // stride over the rows, 16 row loads in flight per lane), combined through the still unused slot buffers, left in the scratch
  // buffer; the CTA that arrives last merges all of them into the running statistics (RunningMeanStd.update_from_moments),
  // refreshes the fp32 (mean, inv_std) and raises the flag every CTA waits for after it has staged its weights -- the merge and
  // the other CTAs' staging overlap, and the separate statistics launch (12 us at 131 072 rows, a latency chain) is gone.
  // All CTAs of the launch are resident together (grid <= SM count, one CTA per SM), so the wait cannot starve anyone.
  if (a.fs_stats) {
    double* sh = reinterpret_cast<double*>(smem + kSmSlot);
    const int w = (int)(tid >> 5);
    const int64_t warp_id = (int64_t)blockIdx.x * (kFwdThreads / 32) + w, n_warps = (int64_t)gridDim.x * (kFwdThreads / 32);
    double s = 0.0, q = 0.0;
    if ((int)lane < obs_dim) {
      for (int64_t i = warp_id; i < a.n; i += 16 * n_warps) {
        float v[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int64_t r = i + k * n_warps;
          v[k] = r < a.n ? __ldg(a.obs + r * a.obs_stride + lane) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 16; k += 2) {
          s += (double)v[k] + (double)v[k + 1];
          q += (double)v[k] * v[k] + (double)v[k + 1] * v[k + 1];
        }
      }
    }
    sh[w * 2 * kStatMaxDim + lane] = s; sh[w * 2 * kStatMaxDim + kStatMaxDim + lane] = q;
    __syncthreads();
    if (tid < 2 * kStatMaxDim) {
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < kFwdThreads / 32; ++k) acc += sh[k * 2 * kStatMaxDim + tid];
      a.fs_scratch[(size_t)blockIdx.x * 2 * kStatMaxDim + tid] = acc;
    }
    unsigned int* words = stat_words(a.fs_scratch);  // [0] ticket, [2] flag, [4] CTAs past the flag
    if (last_block_done(words)) {
      welford_merge_block(a.fs_scratch, (int)gridDim.x, a.n, obs_dim, a.fs_stats, a.fs_eps, a.fs_mean_out, a.fs_inv_out);
      __threadfence();
      __syncthreads();
      if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(words + 2), "r"(1u) : "memory");
    }
    __syncthreads();  // the slot buffers are free again
  }
  // ---- one-time: weights, biases, normalisation constants -> smem; TMEM; barriers
  stage_weight(smem + kSmW1, (const __nv_bfloat16*)a.p.w1, 2 * kHid, kIn, tid, kFwdThreads);
  stage_weight(smem + kSmW2p, (const __nv_bfloat16*)a.p.w2p, kHid, kHid, tid, kFwdThreads);
  stage_weight(smem + kSmW2v, (const __nv_bfloat16*)a.p.w2v, kHid, kHid, tid, kFwdThreads);
  stage_weight(smem + kSmW3, (const __nv_bfloat16*)a.p.w3, kHead, 2 * kHid, tid, kFwdThreads);
  K2_TRACE(125);  // weights staged
  float* sB1 = reinterpret_cast<float*>(smem + kSmB1);
  float* sB2 = reinterpret_cast<float*>(smem + kSmB2);
  float* sB3 = reinterpret_cast<float*>(smem + kSmB3);
  float* sMean = reinterpret_cast<float*>(smem + kSmNorm);
  float* sInv = sMean + kIn;
  if (tid < 2 * kHid) { sB1[tid] = a.p.b1[tid]; sB2[tid] = a.p.b2[tid]; }
  if (tid < kHead) sB3[tid] = a.p.b3[tid];
  if (a.fs_stats) {  // fused statistics, second half: wait for the merged (mean, inv_std); the last CTA through re-arms the words
    unsigned int* words = stat_words(a.fs_scratch);
    if (tid == 0) {
      unsigned int v, ns = 32u;
      while (true) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(words + 2) : "memory");
        if (v != 0u) break;
        __nanosleep(ns);
        if (ns < 256u) ns += ns;
      }
      if (atomicAdd(words + 4, 1u) == gridDim.x - 1) { words[4] = 0u; __threadfence(); words[2] = 0u; }
    }
    __syncthreads();
  }
  // two-launch form of ppo_policy_forward_stats: this grid was scheduled while the statistics kernel was still merging; everything
  // above (weights, biases) does not depend on it, everything below (mean / inv_std, the observations) does
  if (a.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");
  if (tid < kIn) {
    sMean[tid] = (a.obs_mean && (int)tid < obs_dim) ? __ldcg(a.obs_mean + tid) : 0.f;
    sInv[tid] = (a.obs_inv_std && (int)tid < obs_dim) ? __ldcg(a.obs_inv_std + tid) : 1.f;
  }
  if (tid < 32) tmem_alloc(&tmem_slot, kTmemCols);
  if (tid == 0) {
    for (int sidx = 0; sidx < kSlots; ++sidx) mbar_init(&bars[sidx], 1);
    mbar_fence_init();
  }
  K2_TRACE(124);  // biases, TMEM allocation, barrier init
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  K2_TRACE(123);  // CTA-wide sync passed
  uint64_t* bar = &bars[slot];
  const uint32_t tacc = tmem_slot + slot * kSlotTmem;             // MMA destination (lane field 0)
  const uint32_t tacc_row = tacc + (((swarp & 3) * 32u) << 16);   // this warp's lane quarter
  uint8_t* slotp = smem + kSmSlot + slot * kSlotBytes;
  const uint32_t sX = smem_u32(slotp + kSlotX), sH = smem_u32(slotp + kSlotH);
  const uint32_t sW1 = smem_u32(smem + kSmW1), sW2p = smem_u32(smem + kSmW2p), sW2v = smem_u32(smem + kSmW2v), sW3 = smem_u32(smem + kSmW3);
  constexpr uint32_t LBO_ACT = 128 * 16, LBO_W1 = 2 * kHid * 16, LBO_W2 = kHid * 16, LBO_W3 = kHead * 16;
  const uint32_t idesc_h = make_idesc_bf16(128, kHid), idesc_o = make_idesc_bf16(128, kHead);
  uint32_t phase = 0;
  const int64_t n_rows = a.gather_idx ? (int64_t)*a.gather_count : a.n;
  const int n_tiles = (int)((n_rows + 127) / 128);  // 32-bit tile indices (rows stay 64-bit): the kernel sits at its 80-register cap
  const float clipv = a.obs_clip > 0.f ? a.obs_clip : 3.0e38f;
  const uint64_t step = a.step + (a.step_base ? *a.step_base : 0ull);

  long long* dbg = (blockIdx.x == 0 && slot == 0) ? g_phase_clk : nullptr;
  int it = -1;
  // slot-major tile order: tile t belongs to CTA t % grid, so the tiles that do not fill a whole round of grid x kSlots slots are
  // spread over the CTAs (1 024 tiles on 148 SMs: 6 or 7 per SM) instead of giving the first CTAs a third tile in every slot (9 vs 6)
  const int tile_stride = a.grid * kSlots, tile0 = slot * a.grid + (int)blockIdx.x;

  // normalise (VecNormalize.normalize_obs) the raw row chunks in xbuf, write them as bf16 into the slot's X operand
  // (interleaved K-major; 2 threads per row, 2 chunks of 8 columns each) and, if asked, as fp32 into obs_norm_out
  auto stage_x = [&](int64_t tile, const float (&xraw)[16]) {
    const bool xvalid = tile * 128 + xrow < n_rows;
    const int64_t xr = !xvalid ? 0 : (a.gather_idx ? (int64_t)a.gather_idx[tile * 128 + xrow] : tile * 128 + xrow);
#pragma unroll
    for (int qq = 0; qq < 2; ++qq) {
      const int q = 2 * (int)xh + qq, c0 = 8 * q;
      float x[8];
      uint32_t w[4];
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const float v0 = fminf(fmaxf((xraw[8 * qq + 2 * h] - sMean[c0 + 2 * h]) * sInv[c0 + 2 * h], -clipv), clipv);
        const float v1 = fminf(fmaxf((xraw[8 * qq + 2 * h + 1] - sMean[c0 + 2 * h + 1]) * sInv[c0 + 2 * h + 1], -clipv), clipv);
        x[2 * h] = v0; x[2 * h + 1] = v1;
        __nv_bfloat162 pk = __floats2bfloat162_rn(v0, v1);
        w[h] = *reinterpret_cast<uint32_t*>(&pk);
      }
      *reinterpret_cast<uint4*>(slotp + kSlotX + chunk_off(xrow, q, 128)) = make_uint4(w[0], w[1], w[2], w[3]);
      if (a.obs_norm_out && xvalid) {
        float* dst = a.obs_norm_out + xr * obs_dim + c0;
        if (a.norm_vec && c0 + 8 <= obs_dim) {
          *reinterpret_cast<float4*>(dst) = make_float4(x[0], x[1], x[2], x[3]);
          *reinterpret_cast<float4*>(dst + 4) = make_float4(x[4], x[5], x[6], x[7]);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (c0 + j < obs_dim) dst[j] = x[j];
        }
      }
    }
  };
  // last epilogue of a tile: action mean + value out of TMEM, Gaussian sample, log-prob, clipping, global stores
  auto finish_tile = [&](int64_t tile) {
    if (swarp >= 4) return;  // one thread per row
    const bool valid = tile * 128 + erow < n_rows;
    const int64_t row = !valid ? 0 : (a.gather_idx ? (int64_t)a.gather_idx[tile * 128 + erow] : tile * 128 + erow);
    uint32_t r[16];
    tmem_ld16(tacc_row + kTmemOut, r);
    tmem_ld_wait();
    if (!valid) return;
    float mean[4] = {0.f, 0.f, 0.f, 0.f}, act[4] = {0.f, 0.f, 0.f, 0.f}, nz[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < act_dim) mean[j] = __uint_as_float(r[j]) + sB3[j];
    float value = 0.f;
#pragma unroll
    for (int j = 0; j < 5; ++j)
      if (j == act_dim) value = __uint_as_float(r[j]) + sB3[j];
    float logp = 0.f;
    if (!a.deterministic) {
      const uint64_t gid = a.row0 + (uint64_t)row;
      const uint4 b = qx::philox4x32_10(make_uint4(0u, 3u, (uint32_t)step, (uint32_t)(step >> 32)), a.seed_lo ^ (uint32_t)gid,
                                        a.seed_hi ^ (uint32_t)(gid >> 32));
      const float ra = sqrtf(-2.f * __logf(qx::u01(b.x))), rb = sqrtf(-2.f * __logf(qx::u01(b.z)));
      float s0, c0, s1, c1;
      __sincosf(6.28318530718f * qx::u01(b.y) - 3.14159265359f, &s0, &c0);
      __sincosf(6.28318530718f * qx::u01(b.w) - 3.14159265359f, &s1, &c1);
      nz[0] = -ra * c0; nz[1] = -ra * s0; nz[2] = -rb * c1; nz[3] = -rb * s1;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (j < act_dim) {
        const float ls = __ldg(a.p.log_std + j);
        act[j] = fmaf(__expf(ls), nz[j], mean[j]);
        logp += -0.5f * nz[j] * nz[j] - ls - 0.91893853320467f;
      }
    if (a.act_vec) {
      if (a.actions) *reinterpret_cast<float4*>(a.actions + row * 4) = make_float4(act[0], act[1], act[2], act[3]);
      if (a.env_actions)
        *reinterpret_cast<float4*>(a.env_actions + row * 4) =
            make_float4(qx::clampf(act[0], -1.f, 1.f), qx::clampf(act[1], -1.f, 1.f), qx::clampf(act[2], -1.f, 1.f), qx::clampf(act[3], -1.f, 1.f));
    } else {
      for (int j = 0; j < act_dim; ++j) {
        if (a.actions) a.actions[row * act_dim + j] = act[j];
        if (a.env_actions) a.env_actions[row * act_dim + j] = qx::clampf(act[j], -1.f, 1.f);
      }
    }
    if (a.values) a.values[row] = value;
    if (a.log_probs) a.log_probs[row] = logp;
    if (a.boot_reward && a.boot_tr[row] && !a.boot_te[row])
      a.boot_reward[row] = a.boot_store ? a.boot_gamma * value : fmaf(a.boot_gamma, value, a.boot_reward[row]);
  };
  auto issue_l1p = [&]() {
#pragma unroll
    for (int ks = 0; ks < kIn / 16; ++ks)
      mma_bf16(tacc, make_desc(sX + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW1 + ks * 2 * LBO_W1, LBO_W1, 128), idesc_h, ks > 0);
  };

  // Software pipeline over this slot's tiles.  Commit groups per tile i:
  //   G_a = {L3v(i-1), L1p(i)}   G_b = {L2p(i)}   G_c = {L3p(i), L1v(i)}   G_d = {L2v(i)}
  // The X operand of tile i+1 is staged (from registers prefetched one tile earlier) right after G_c(i) released X,
  // so neither its global-memory latency nor the global stores (obs_norm_out, actions, ...) sit between a
  // fence.proxy.async and the barrier that precedes an MMA issue.
  if (tile0 < n_tiles) {
    float xbuf[16];
    K2_TRACE(122);  // per-slot setup
    load_obs_chunks(a, tile0, n_rows, xrow, xh, obs_dim, xbuf);
    stage_x(tile0, xbuf);
    K2_TRACE(121);  // first X tile loaded + staged
    load_obs_chunks(a, tile0 + tile_stride, n_rows, xrow, xh, obs_dim, xbuf);
    fence_async_smem();
    fence_before_sync();
    slot_sync(slot);
    if (st == 0) { fence_after_sync(); issue_l1p(); mma_commit(bar); }
    int64_t prev = -1;
    for (int tile = tile0; tile < n_tiles; tile += tile_stride) {
      ++it;
      PHASE_STAMP(0);
      // ---- G_a: action/value of the previous tile are complete, and this tile's actor layer 1
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      PHASE_STAMP(1);
      if (prev >= 0) finish_tile(prev);
      hidden_epilogue(tacc_row, sB1, slotp + kSlotH, erow, ecol0);
      fence_async_smem();
      fence_before_sync();
      slot_sync(slot);
      PHASE_STAMP(2);
      // ---- G_b = [L2p]
      if (st == 0) {
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < kHid / 16; ++ks)
          mma_bf16(tacc, make_desc(sH + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW2p + ks * 2 * LBO_W2, LBO_W2, 128), idesc_h, ks > 0);
        mma_commit(bar);
      }
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      PHASE_STAMP(3);
      hidden_epilogue(tacc_row, sB2, slotp + kSlotH, erow, ecol0);
      fence_async_smem();
      fence_before_sync();
      slot_sync(slot);
      PHASE_STAMP(4);
      // ---- G_c = [L3p, L1v]: action head from H2p into the out columns; critic layer 1 from X into the accumulator
      if (st == 0) {
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < kHid / 16; ++ks)
          mma_bf16(tacc + kTmemOut, make_desc(sH + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW3 + ks * 2 * LBO_W3, LBO_W3, 128), idesc_o, ks > 0);
#pragma unroll
        for (int ks = 0; ks < kIn / 16; ++ks)
          mma_bf16(tacc, make_desc(sX + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW1 + kHid * 16 + ks * 2 * LBO_W1, LBO_W1, 128), idesc_h, ks > 0);
        mma_commit(bar);
      }
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      PHASE_STAMP(5);
      // X is free: stage the next tile (its raw rows are in xbuf) and request the one after
      const int next = tile + tile_stride;
      if (next < n_tiles) {
        stage_x(next, xbuf);
        load_obs_chunks(a, next + tile_stride, n_rows, xrow, xh, obs_dim, xbuf);
      }
      hidden_epilogue(tacc_row, sB1 + kHid, slotp + kSlotH, erow, ecol0);
      fence_async_smem();
      fence_before_sync();
      slot_sync(slot);
      PHASE_STAMP(6);
      // ---- G_d = [L2v]
      if (st == 0) {
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < kHid / 16; ++ks)
          mma_bf16(tacc, make_desc(sH + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW2v + ks * 2 * LBO_W2, LBO_W2, 128), idesc_h, ks > 0);
        mma_commit(bar);
      }
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      PHASE_STAMP(7);
      hidden_epilogue(tacc_row, sB2 + kHid, slotp + kSlotH, erow, ecol0);
      fence_async_smem();
      fence_before_sync();
      slot_sync(slot);
      PHASE_STAMP(8);
      // ---- G_a of the next tile = [L3v (value head accumulated onto the action-head result), L1p(next)]
      if (st == 0) {
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < kHid / 16; ++ks)
          mma_bf16(tacc + kTmemOut, make_desc(sH + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW3 + (16 + ks * 2) * LBO_W3, LBO_W3, 128), idesc_o, true);
        if (next < n_tiles) issue_l1p();
        mma_commit(bar);
      }
      prev = tile;
      PHASE_STAMP(9);
    }
    mbar_wait(bar, phase); phase ^= 1;
    fence_after_sync();
    finish_tile(prev);
    fence_before_sync();
  }
  __syncthreads();
  K2_TRACE(126);
  if (tid < 32) tmem_dealloc(tmem_slot, kTmemCols);
}

// ---------------------------------------------------------------------------
// K3: GAE(lambda) -- RolloutBuffer.compute_returns_and_advantage.  One thread per
// env walks its column of the [T, n] buffers backwards (coalesced across envs):
//   delta_t = r_t + gamma V_{t+1} (1 - d_t) - V_t ;  A_t = delta_t + gamma lam (1 - d_t) A_{t+1}
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gae_kernel(const float* __restrict__ rew, const float* __restrict__ val, const uint8_t* __restrict__ done,
                                                  const float* __restrict__ last_val, int T, int64_t n, float gamma, float lam,
                                                  float* __restrict__ adv, float* __restrict__ ret) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float next_v = last_val[i], gae = 0.f;
  // software pipeline: the loads of step t-1 are issued before the arithmetic of step t
  float r = rew[(int64_t)(T - 1) * n + i], v = val[(int64_t)(T - 1) * n + i];
  uint8_t d = done[(int64_t)(T - 1) * n + i];
  for (int t = T - 1; t >= 0; --t) {
    float r2 = 0.f, v2 = 0.f;
    uint8_t d2 = 0;
    if (t > 0) { r2 = rew[(int64_t)(t - 1) * n + i]; v2 = val[(int64_t)(t - 1) * n + i]; d2 = done[(int64_t)(t - 1) * n + i]; }
    const float nnt = d ? 0.f : 1.f;
    const float delta = fmaf(gamma * next_v, nnt, r) - v;
    gae = fmaf(gamma * lam * nnt, gae, delta);
    adv[(int64_t)t * n + i] = gae;
    ret[(int64_t)t * n + i] = gae + v;
    next_v = v;
    r = r2; v = v2; d = d2;
  }
}

// K3b: the same recurrence as a warp scan over time, for batches too small to fill the GPU with one thread per env.
// A block owns 32 envs; per 32-step time tile (walked from the end) warp w loads row t0 + w coalesced across its 32
// envs, the tile is transposed through shared memory so that warp w holds env w with lane = time, and the affine maps
// x -> delta_t + c_t x (c_t = gamma lam (1 - d_t)) are composed by a 5-round Kogge-Stone suffix scan with
// __shfl_down_sync; the carry into the tile is the advantage at the start of the previously processed tile.
constexpr int kScanTile = 32;
__global__ void __launch_bounds__(1024) gae_warpscan_kernel(const float* __restrict__ rew, const float* __restrict__ val, const uint8_t* __restrict__ done,
                                                           const float* __restrict__ last_val, int T, int64_t n, float gamma, float lam,
                                                           float* __restrict__ adv, float* __restrict__ ret) {
  __shared__ float sV[kScanTile + 1][kScanTile + 1], sD[kScanTile][kScanTile + 1], sC[kScanTile][kScanTile + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t e0 = (int64_t)blockIdx.x * kScanTile;
  const int64_t env_row = e0 + lane;   // load / store phase: lane = env, warp = time
  const bool env_ok = env_row < n;
  float carry = 0.f;                   // scan phase: warp = env; advantage at the first step of the tile processed before
  const int n_tiles = (T + kScanTile - 1) / kScanTile;
  for (int tile = n_tiles - 1; tile >= 0; --tile) {
    const int t0 = tile * kScanTile, t = t0 + w;
    const bool ok = env_ok && t < T;
    float r = 0.f, v = 0.f, nnt = 1.f;
    if (ok) {
      r = rew[(int64_t)t * n + env_row]; v = val[(int64_t)t * n + env_row];
      nnt = done[(int64_t)t * n + env_row] ? 0.f : 1.f;
    }
    sV[w][lane] = v;
    if (w == 0) {  // row t0 + 32: value after the tile (the rollout's last_values for the final tile)
      const int tn = t0 + kScanTile;
      sV[kScanTile][lane] = !env_ok ? 0.f : (tn < T ? val[(int64_t)tn * n + env_row] : last_val[env_row]);
    }
    __syncthreads();
    // value of the next step: next row of the tile, or last_values right after the final step of the rollout
    const float vn = (t + 1 < T) ? sV[w + 1][lane] : (env_ok ? last_val[env_row] : 0.f);
    sD[w][lane] = ok ? fmaf(gamma * vn, nnt, r) - v : 0.f;   // delta_t; steps past T are the identity map
    sC[w][lane] = ok ? gamma * lam * nnt : 1.f;
    __syncthreads();
    // transposed: warp w = env e0 + w, lane = time t0 + lane
    float d = sD[lane][w], c = sC[lane][w];
#pragma unroll
    for (int off = 1; off < kScanTile; off <<= 1) {
      const float d2 = __shfl_down_sync(0xffffffffu, d, off), c2 = __shfl_down_sync(0xffffffffu, c, off);
      if (lane + off < kScanTile) { d = fmaf(c, d2, d); c *= c2; }
    }
    const float a = fmaf(c, carry, d);
    carry = __shfl_sync(0xffffffffu, a, 0);
    __syncthreads();
    sD[lane][w] = a;
    __syncthreads();
    if (ok) {
      const float av = sD[w][lane];
      adv[(int64_t)t * n + env_row] = av;
      ret[(int64_t)t * n + env_row] = av + v;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// K4: VecNormalize running statistics, one launch: every block leaves fp64 sums
// of x and x^2 per column in the scratch buffer; the block that finishes last
// (a ticket in the tail of the scratch buffer) turns them into batch moments
// and does the parallel-Welford merge into {mean[dim], var[dim], count}, and
// refreshes the fp32 mean / inv_std the policy kernel reads.
// ---------------------------------------------------------------------------
constexpr int kStatBlocks = 148, kStatThreads = 1024, kRetThreads = 1024;  // one wave of full-SM blocks (kStatMaxDim = 32: above)
constexpr size_t kStatTicketOffset = (size_t)kStatBlocks * 2 * kStatMaxDim;  // in doubles
// the 16 32-bit words behind the partial sums: [0] last-block ticket; the fused policy launch also uses [2] and [4]
__device__ __forceinline__ unsigned int* stat_words(double* scratch) { return reinterpret_cast<unsigned int*>(scratch + kStatTicketOffset); }

// true in exactly one block per launch: the last one to arrive; it re-arms the ticket for the next launch / graph replay
__device__ __forceinline__ bool last_block_done(unsigned int* ticket) {
  __shared__ bool is_last;
  __threadfence();  // this block's partial sums are visible device-wide before its ticket is
  __syncthreads();
  if (threadIdx.x == 0) {
    is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    if (is_last) *ticket = 0u;
  }
  __syncthreads();
  if (is_last) __threadfence();
  return is_last;
}

// one warp per column: lanes stride over the per-block partial sums (at most kStatBlocks / 32 = 5 each, all loads issued
// before the first add), shuffle-reduce, lane 0 does the Welford merge
__device__ __forceinline__ void welford_merge_block(const double* part, int nblocks, int64_t n, int dim, double* __restrict__ stats, float eps,
                                                    float* __restrict__ mean_f32, float* __restrict__ inv_std_f32) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const double count = stats[2 * dim], bc = (double)n, tot = count + bc;
  const double inv_bc = 1.0 / bc, inv_tot = 1.0 / tot;
  __syncthreads();  // every warp has the old count before thread 0 replaces it
  constexpr int kPer = (kStatBlocks + 31) / 32;
  for (int j = w; j < dim; j += nw) {
    double sv[kPer], qv[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int b = lane + 32 * k;
      sv[k] = b < nblocks ? __ldcg(part + (size_t)b * 2 * kStatMaxDim + j) : 0.0;
      qv[k] = b < nblocks ? __ldcg(part + (size_t)b * 2 * kStatMaxDim + kStatMaxDim + j) : 0.0;
    }
    double s = 0.0, q = 0.0;
#pragma unroll
    for (int k = 0; k < kPer; ++k) { s += sv[k]; q += qv[k]; }
    for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
    if (lane == 0) {
      const double bm = s * inv_bc, bv = fmax(q * inv_bc - bm * bm, 0.0);
      const double mean = stats[j], var = stats[dim + j];
      const double delta = bm - mean;
      const double new_mean = mean + delta * bc * inv_tot;
      const double new_var = (var * count + bv * bc + delta * delta * count * bc * inv_tot) * inv_tot;
      stats[j] = new_mean;
      stats[dim + j] = new_var;
      if (mean_f32) mean_f32[j] = (float)new_mean;
      if (inv_std_f32) inv_std_f32[j] = (float)(1.0 / sqrt(new_var + (double)eps));
    }
  }
  if (threadIdx.x == 0) stats[2 * dim] = tot;
}

// lane = column (dim <= 32), each warp strides over rows: a row is one coalesced load, no cross-lane reduction is needed;
// 32 warps per block keep enough loads in flight (the kernel is latency-, not bandwidth-bound: 10 MB at 131 072 x 20);
// the warps of a block are combined through shared memory
__global__ void __launch_bounds__(kStatThreads) running_stats_kernel(const float* __restrict__ x, int64_t stride, int64_t n, int dim,
                                                                    double* __restrict__ scratch, double* __restrict__ stats, float eps,
                                                                    float* __restrict__ mean_f32, float* __restrict__ inv_std_f32) {
  __shared__ double sh[kStatThreads / 32][2 * kStatMaxDim];
  asm volatile("griddepcontrol.launch_dependents;");  // a policy-forward launch chained behind this one may take the SMs as the blocks leave
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t warp_id = (int64_t)blockIdx.x * (kStatThreads / 32) + w, n_warps = (int64_t)gridDim.x * (kStatThreads / 32);
  double s = 0.0, q = 0.0;
  if (lane < dim) {
    // 16 independent row loads in flight per lane: at 131 072 rows over 148 x 32 warps that is two trips to L2 / HBM in all
    for (int64_t i = warp_id; i < n; i += 16 * n_warps) {
      float v[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const int64_t r = i + k * n_warps;
        v[k] = r < n ? x[r * stride + lane] : 0.f;
      }
#pragma unroll
      for (int k = 0; k < 16; k += 2) {
        s += (double)v[k] + (double)v[k + 1];
        q += (double)v[k] * v[k] + (double)v[k + 1] * v[k + 1];
      }
    }
  }
  sh[w][lane] = s; sh[w][kStatMaxDim + lane] = q;
  __syncthreads();
  if (threadIdx.x < 2 * kStatMaxDim) {
    double a = 0.0;
#pragma unroll
    for (int k = 0; k < kStatThreads / 32; ++k) a += sh[k][threadIdx.x];
    scratch[(size_t)blockIdx.x * 2 * kStatMaxDim + threadIdx.x] = a;
  }
  if (last_block_done(reinterpret_cast<unsigned int*>(scratch + kStatTicketOffset)))
    welford_merge_block(scratch, (int)gridDim.x, n, dim, stats, eps, mean_f32, inv_std_f32);
}

// reward path, first half fused: ret = ret * gamma + r (VecNormalize.step_wait), the per-block sums of ret, ret^2, and -- in
// the block that finishes last -- the merge into the running variance of the discounted return
__global__ void __launch_bounds__(kRetThreads) returns_stats_kernel(const float* __restrict__ r, float* __restrict__ acc, int64_t n, float gamma,
                                                                   double* __restrict__ scratch, double* __restrict__ ret_stats, float eps) {
  __shared__ double sh[kRetThreads / 32][2];
  double s = 0.0, q = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * kRetThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kRetThreads) {
    const float v = fmaf(acc[i], gamma, r[i]);
    acc[i] = v;
    s += (double)v; q += (double)v * (double)v;
  }
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { sh[w][0] = s; sh[w][1] = q; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double a = 0.0;
    for (int k = 0; k < kRetThreads / 32; ++k) a += sh[k][threadIdx.x];
    scratch[(size_t)blockIdx.x * 2 * kStatMaxDim + (threadIdx.x ? kStatMaxDim : 0)] = a;
  }
  if (last_block_done(reinterpret_cast<unsigned int*>(scratch + kStatTicketOffset)))
    welford_merge_block(scratch, (int)gridDim.x, n, 1, ret_stats, eps, nullptr, nullptr);
}

__global__ void __launch_bounds__(256) reward_norm_kernel(const float* __restrict__ r, const uint8_t* __restrict__ te, const uint8_t* __restrict__ tr, float* __restrict__ acc,
                                                          int64_t n, float clip, float eps, const double* __restrict__ ret_stats, float* out,
                                                          uint8_t* __restrict__ done_out, int add_boot) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float inv = ret_stats ? (float)(1.0 / sqrt(ret_stats[1] + (double)eps)) : 1.f;
  // add_boot: the time-limit bootstrap ran first and left gamma V(terminal_obs) in out[i] for the truncated rows
  const float boot = (add_boot && tr[i] && !te[i]) ? out[i] : 0.f;
  out[i] = fminf(fmaxf(r[i] * inv, -clip), clip) + boot;
  const uint8_t d = te[i] | tr[i];
  if (d && acc) acc[i] = 0.f;
  if (done_out) done_out[i] = d;
}

}  // namespace ppo

static int pfail(int code, const char* msg) { return qx_fail(code, "%s", msg); }

extern "C" int ppo_test_gemm(const void* a, const void* b, float* d, int32_t n, int32_t k, void* stream) {
  if (!a || !b || !d || n < 16 || n > 256 || n % 16 || k < 16 || k % 16) return pfail(QX_EINVAL, "ppo_test_gemm: bad arguments");
  const size_t smem = (size_t)(128 + n) * k * 2;
  if (smem > 200 * 1024) return pfail(QX_EINVAL, "ppo_test_gemm: tile too large");
  cudaFuncSetAttribute(ppo::test_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  ppo::test_gemm_kernel<<<1, 128, smem, (cudaStream_t)stream>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, d, n, k);
  return cudaGetLastError() == cudaSuccess ? QX_OK : pfail(QX_ECUDA, "ppo_test_gemm: launch failed");
}

extern "C" int ppo_test_tanh_bf16(const float* x, uint16_t* out, int64_t n, void* stream) {
  if (!x || !out || n <= 0) return pfail(QX_EINVAL, "ppo_test_tanh_bf16: bad arguments");
  const int64_t pairs = (n + 1) / 2;
  ppo::test_tanh_kernel<<<(unsigned)((pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, n);
  return cudaGetLastError() == cudaSuccess ? QX_OK : pfail(QX_ECUDA, "ppo_test_tanh_bf16: launch failed");
}

static bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

static int launch_forward(ppo::FwdArgs& a, int64_t max_rows, void* stream) {
  a.obs_vec = aligned16(a.obs) && (a.obs_stride & 3) == 0;
  a.norm_vec = (a.p.obs_dim & 3) == 0 && aligned16(a.obs_norm_out);
  a.act_vec = a.p.act_dim == 4 && aligned16(a.actions) && aligned16(a.env_actions);  // (a null pointer is aligned)
  // per device: SM count and the one-time opt-in to ~200 KB of dynamic shared memory (the attribute is per device; the cached
  // value is set only after the call succeeded, so a failure is retried)
  static std::atomic<int> sms_of[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return pfail(QX_ECUDA, "ppo_policy_forward: cannot query the current device");
  int sms = sms_of[dev].load(std::memory_order_acquire);
  if (!sms) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      return pfail(QX_ECUDA, "ppo_policy_forward: cannot query the SM count");
    if (cudaFuncSetAttribute(ppo::policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ppo::kSmTotal) != cudaSuccess)
      return pfail(QX_ECUDA, "ppo_policy_forward: cannot reserve shared memory");
    sms_of[dev].store(n, std::memory_order_release);
    sms = n;
  }
  const int64_t tiles = (max_rows + 127) / 128;
  const unsigned grid = (unsigned)(tiles < sms ? (tiles > 0 ? tiles : 1) : sms);  // small batches: one tile per SM before a second slot is used
  a.grid = (int32_t)grid;
  if (a.pdl_wait) {
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(ppo::kFwdThreads); lc.dynamicSmemBytes = ppo::kSmTotal; lc.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = &at; lc.numAttrs = 1;
    if (cudaLaunchKernelEx(&lc, ppo::policy_forward_kernel, a) != cudaSuccess) return pfail(QX_ECUDA, "ppo_policy_forward: launch failed");
    return QX_OK;
  }
  ppo::policy_forward_kernel<<<grid, ppo::kFwdThreads, ppo::kSmTotal, (cudaStream_t)stream>>>(a);
  return cudaGetLastError() == cudaSuccess ? QX_OK : pfail(QX_ECUDA, "ppo_policy_forward: launch failed");
}

static bool policy_ok(const PpoPolicy* p) {
  return p && p->w1 && p->w2p && p->w2v && p->w3 && p->b1 && p->b2 && p->b3 && p->log_std && p->obs_dim >= 1 && p->obs_dim <= PPO_IN_PAD &&
         p->act_dim >= 1 && p->act_dim <= 4;
}

extern "C" int ppo_policy_forward(const PpoPolicy* p, const float* obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                                  const float* obs_inv_std, float obs_clip, uint64_t seed, uint64_t row0, uint64_t step,
                                  const uint64_t* step_base_dev, int32_t deterministic, float* actions, float* env_actions, float* values,
                                  float* log_probs, float* obs_norm_out, void* stream) {
  if (!policy_ok(p) || !obs || n <= 0 || obs_stride < p->obs_dim) return pfail(QX_EINVAL, "ppo_policy_forward: bad arguments");
  ppo::FwdArgs a{};
  a.p = *p; a.obs = obs; a.obs_stride = obs_stride; a.n = n; a.obs_mean = obs_mean; a.obs_inv_std = obs_inv_std; a.obs_clip = obs_clip;
  a.seed_lo = (uint32_t)seed; a.seed_hi = (uint32_t)(seed >> 32); a.row0 = row0; a.step = step; a.step_base = step_base_dev;
  a.deterministic = deterministic; a.actions = actions; a.env_actions = env_actions; a.values = values; a.log_probs = log_probs;
  a.obs_norm_out = obs_norm_out;
  return launch_forward(a, n, stream);
}

extern "C" int ppo_policy_forward_stats(const PpoPolicy* p, const float* obs, int64_t obs_stride, int64_t n, double* obs_stats, float eps,
                                        void* stats_scratch, float* obs_mean, float* obs_inv_std, float obs_clip, uint64_t seed, uint64_t row0,
                                        uint64_t step, const uint64_t* step_base_dev, int32_t deterministic, float* actions, float* env_actions,
                                        float* values, float* log_probs, float* obs_norm_out, int32_t fused, void* stream) {
  if (!policy_ok(p) || !obs || n <= 0 || obs_stride < p->obs_dim || !obs_stats || !stats_scratch || !obs_mean || !obs_inv_std)
    return pfail(QX_EINVAL, "ppo_policy_forward_stats: bad arguments");
  ppo::FwdArgs a{};
  a.p = *p; a.obs = obs; a.obs_stride = obs_stride; a.n = n; a.obs_mean = obs_mean; a.obs_inv_std = obs_inv_std; a.obs_clip = obs_clip;
  a.seed_lo = (uint32_t)seed; a.seed_hi = (uint32_t)(seed >> 32); a.row0 = row0; a.step = step; a.step_base = step_base_dev;
  a.deterministic = deterministic; a.actions = actions; a.env_actions = env_actions; a.values = values; a.log_probs = log_probs;
  a.obs_norm_out = obs_norm_out;
  if (fused) {
    a.fs_stats = obs_stats; a.fs_scratch = (double*)stats_scratch; a.fs_eps = eps; a.fs_mean_out = obs_mean; a.fs_inv_out = obs_inv_std;
    return launch_forward(a, n, stream);
  }
  // two launches, the second a programmatic dependent of the first: the policy kernel stages its weights while the statistics
  // kernel's last block still merges, and waits on the device before it reads (mean, inv_std)
  int rc = ppo_running_stats_update(obs, obs_stride, n, p->obs_dim, obs_stats, eps, obs_mean, obs_inv_std, stats_scratch, stream);
  if (rc) return rc;
  a.pdl_wait = 1;
  return launch_forward(a, n, stream);
}

extern "C" int ppo_bootstrap_truncated(const PpoPolicy* p, const float* terminal_obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                                       const float* obs_inv_std, float obs_clip, const uint32_t* done_count_dev, const uint32_t* done_idx_dev,
                                       const uint8_t* terminated, const uint8_t* truncated, float gamma, float* reward_inout, void* stream) {
  if (!policy_ok(p) || !terminal_obs || n <= 0 || !done_count_dev || !done_idx_dev || !terminated || !truncated || !reward_inout)
    return pfail(QX_EINVAL, "ppo_bootstrap_truncated: bad arguments");
  ppo::FwdArgs a{};
  a.p = *p; a.obs = terminal_obs; a.obs_stride = obs_stride; a.n = n; a.obs_mean = obs_mean; a.obs_inv_std = obs_inv_std; a.obs_clip = obs_clip;
  a.deterministic = 1; a.gather_idx = done_idx_dev; a.gather_count = done_count_dev; a.boot_reward = reward_inout; a.boot_te = terminated;
  a.boot_tr = truncated; a.boot_gamma = gamma;
  return launch_forward(a, n, stream);
}

extern "C" int ppo_bootstrap_truncated_first(const PpoPolicy* p, const float* terminal_obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                                             const float* obs_inv_std, float obs_clip, const uint32_t* done_count_dev, const uint32_t* done_idx_dev,
                                             const uint8_t* terminated, const uint8_t* truncated, float gamma, float* reward_out, void* stream) {
  if (!policy_ok(p) || !terminal_obs || n <= 0 || !done_count_dev || !done_idx_dev || !terminated || !truncated || !reward_out)
    return pfail(QX_EINVAL, "ppo_bootstrap_truncated_first: bad arguments");
  ppo::FwdArgs a{};
  a.p = *p; a.obs = terminal_obs; a.obs_stride = obs_stride; a.n = n; a.obs_mean = obs_mean; a.obs_inv_std = obs_inv_std; a.obs_clip = obs_clip;
  a.deterministic = 1; a.gather_idx = done_idx_dev; a.gather_count = done_count_dev; a.boot_reward = reward_out; a.boot_te = terminated;
  a.boot_tr = truncated; a.boot_gamma = gamma; a.boot_store = 1;
  return launch_forward(a, n, stream);
}

extern "C" int ppo_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, int32_t T, int64_t n,
                       float gamma, float lam, float* advantages, float* returns, void* stream) {
  if (!rewards || !values || !dones || !last_values || !advantages || !returns || T <= 0 || n <= 0) return pfail(QX_EINVAL, "ppo_gae: bad arguments");
  // one thread per env saturates the memory system once there are enough envs; below that, scan over time in warps
  if (n >= (1 << 17) || T < 16)
    ppo::gae_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, T, n, gamma, lam, advantages, returns);
  else
    ppo::gae_warpscan_kernel<<<(unsigned)((n + ppo::kScanTile - 1) / ppo::kScanTile), 1024, 0, (cudaStream_t)stream>>>(rewards, values, dones, last_values, T,
                                                                                                                       n, gamma, lam, advantages, returns);
  return cudaGetLastError() == cudaSuccess ? QX_OK : pfail(QX_ECUDA, "ppo_gae: launch failed");
}

extern "C" int64_t ppo_running_stats_scratch_bytes(int32_t dim) {
  (void)dim;
  return (int64_t)(ppo::kStatTicketOffset + 8) * sizeof(double);  // per-block partial sums + the last-block ticket
}

extern "C" int ppo_running_stats_update(const float* x, int64_t stride, int64_t n, int32_t dim, double* stats, float eps, float* mean_f32,
                                        float* inv_std_f32, void* scratch, void* stream) {
  if (!x || !stats || !scratch || n <= 0 || dim < 1 || dim > ppo::kStatMaxDim || stride < dim) return pfail(QX_EINVAL, "ppo_running_stats_update: bad arguments");
  int64_t want = (n + ppo::kStatThreads / 32 * 8 - 1) / (ppo::kStatThreads / 32 * 8);  // >= 8 rows per warp
  const int blocks = (int)(want < ppo::kStatBlocks ? (want < 1 ? 1 : want) : ppo::kStatBlocks);
  ppo::running_stats_kernel<<<blocks, ppo::kStatThreads, 0, (cudaStream_t)stream>>>(x, stride, n, dim, (double*)scratch, stats, eps, mean_f32, inv_std_f32);
  return cudaGetLastError() == cudaSuccess ? QX_OK : pfail(QX_ECUDA, "ppo_running_stats_update: launch failed");
}

static int reward_normalize_impl(const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns_acc, int64_t n,
                                 float gamma, float clip, float eps, double* ret_stats, float* reward_out, uint8_t* done_out, void* scratch, void* stream,
                                 int add_boot) {
  if (!reward || !terminated || !truncated || !returns_acc || !ret_stats || !reward_out || !scratch || n <= 0)
    return pfail(QX_EINVAL, "ppo_reward_normalize: bad arguments");
  const unsigned grid = (unsigned)((n + 255) / 256);
  int64_t want = (n + ppo::kRetThreads - 1) / ppo::kRetThreads;
  const int blocks = (int)(want < ppo::kStatBlocks ? want : ppo::kStatBlocks);
  ppo::returns_stats_kernel<<<blocks, ppo::kRetThreads, 0, (cudaStream_t)stream>>>(reward, returns_acc, n, gamma, (double*)scratch, ret_stats, eps);
  ppo::reward_norm_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(reward, terminated, truncated, returns_acc, n, clip, eps, ret_stats, reward_out, done_out, add_boot);
  return cudaGetLastError() == cudaSuccess ? QX_OK : pfail(QX_ECUDA, "ppo_reward_normalize: launch failed");
}

extern "C" int ppo_reward_normalize(const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns_acc, int64_t n,
                                    float gamma, float clip, float eps, double* ret_stats, float* reward_out, uint8_t* done_out, void* scratch, void* stream) {
  return reward_normalize_impl(reward, terminated, truncated, returns_acc, n, gamma, clip, eps, ret_stats, reward_out, done_out, scratch, stream, 0);
}

extern "C" int ppo_reward_normalize_add(const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns_acc, int64_t n,
                                        float gamma, float clip, float eps, double* ret_stats, float* reward_out, uint8_t* done_out, void* scratch,
                                        void* stream) {
  return reward_normalize_impl(reward, terminated, truncated, returns_acc, n, gamma, clip, eps, ret_stats, reward_out, done_out, scratch, stream, 1);
}

// debug / tuning hook (not part of the public header): device buffer of 8 x 16 int64 clock stamps, or NULL to switch off
extern "C" int ppo_debug_phase_clock(long long* dev_buf) {
  return cudaMemcpyToSymbol(ppo::g_phase_clk, &dev_buf, sizeof(dev_buf)) == cudaSuccess ? QX_OK : QX_ECUDA;
}
