// sac_kernels.cu -- stable-baselines3 SAC actor forward for sm_100a (C-ABI: include/sac_b200.h).
//   K8  deterministic SAC actor (ReLU MLP + tanh squash) on tcgen05 tensor cores, fused VecNormalize
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <climits>

#include "../../include/quadx_b200.h"
#include "../../include/sac_b200.h"
#include "qx_internal.h"
#include "tc05.cuh"

namespace sac {

using namespace tc05;

// ---------------------------------------------------------------------------
// K8: SB3 Actor in deterministic mode.  Persistent CTAs, one per SM, 512 threads = four independent slots of 128
// threads (one warpgroup: warp w of a slot reads TMEM lanes 32 w .. 32 w + 31, so thread = tile row throughout).
// Each slot walks its own 128-row tiles in slot-major order; per tile
//   [L1]  X[128x32]  . W1^T    -> acc (TMEM, the slot's 128 columns)   then bias + ReLU + bf16 -> H
//   [L2]  H[128x128] . W2^T    -> acc                                  then bias + ReLU + bf16 -> H (in place)
//   [L3]  H          . Wmu^T   -> acc columns 0..15                    then bias + tanh -> actions
// Each [..] is one commit -> mbarrier wait.  The X operand of the next tile is staged as soon as L1 has released it
// (its raw rows were loaded into registers one tile earlier).  Weights (44 KB bf16) stay resident in shared memory.
// Four slots x 128 TMEM columns fill the 512 columns; a slot's three MMA groups are sequential, the other slots' epilogues
// run meanwhile.
// ---------------------------------------------------------------------------
constexpr int kHid = SAC_HIDDEN, kIn = SAC_IN_PAD, kHead = SAC_HEAD_PAD;
constexpr int kSlots = 4, kSlotThreads = 128, kThreads = kSlots * kSlotThreads;
constexpr uint32_t kSmW1 = 0;                                   // [4][128][16 B]
constexpr uint32_t kSmW2 = kSmW1 + kHid * kIn * 2;              // [16][128][16 B]
constexpr uint32_t kSmWmu = kSmW2 + kHid * kHid * 2;            // [16][16][16 B]
constexpr uint32_t kSmSlot = kSmWmu + kHead * kHid * 2;         // per slot: X [4][128][16 B] then H [16][128][16 B]
constexpr uint32_t kSlotX = 0, kSlotH = 128 * kIn * 2, kSlotBytes = kSlotH + 128 * kHid * 2;
constexpr uint32_t kSmB1 = kSmSlot + kSlots * kSlotBytes;       // 128 f32
constexpr uint32_t kSmB2 = kSmB1 + kHid * 4;                    // 128 f32
constexpr uint32_t kSmBmu = kSmB2 + kHid * 4;                   // 16 f32
constexpr uint32_t kSmNorm = kSmBmu + kHead * 4;                // mean[32], inv_std[32]
constexpr uint32_t kSmTotal = kSmNorm + 2 * kIn * 4;
constexpr uint32_t kTmemCols = 512, kSlotTmem = kHid;
static_assert(kSlots * kSlotTmem <= kTmemCols && kSmTotal <= 227 * 1024, "slots must fit TMEM and shared memory");

struct Args {
  SacActor p;
  const float* obs;
  int64_t obs_stride, n;
  const float* obs_mean;
  const float* obs_inv_std;
  float obs_clip;
  float* actions;
  float* obs_norm_out;
  int32_t grid;      // CTAs of this launch (= gridDim.x)
  // 16-byte vector paths, decided on the host so that the branches are uniform
  int32_t obs_vec;   // obs rows as float4: obs 16-byte aligned and obs_stride % 4 == 0
  int32_t norm_vec;  // obs_norm_out rows as float4: obs_norm_out 16-byte aligned and obs_dim % 4 == 0
  int32_t act_vec;   // actions rows as float4: act_dim == 4 and actions 16-byte aligned
};

__device__ __forceinline__ uint32_t relu_pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
  return *reinterpret_cast<uint32_t*>(&v);
}

// tanh rounded from fp64: --use_fast_math turns tanhf into tanh.approx.f32 (MUFU.TANH, ~2^-11 relative), and a reference
// should restate the squash as np.tanh without a hook of the kernel.  Four per row: the fp64 cost is negligible.
__device__ __forceinline__ float accurate_tanh(float x) { return (float)tanh((double)x); }

// bias + ReLU + bf16 of the 128 accumulator columns of this thread's row -> H chunks (A operand of the next layer)
__device__ __forceinline__ void relu_epilogue(uint32_t tacc_row, const float* __restrict__ bias, uint8_t* sH, uint32_t row) {
#pragma unroll
  for (int c0 = 0; c0 < kHid; c0 += 32) {
    uint32_t r[32];
    tmem_ld32(tacc_row + c0, r);
    tmem_ld_wait();
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 b0 = *reinterpret_cast<const float4*>(bias + c0 + 8 * q), b1 = *reinterpret_cast<const float4*>(bias + c0 + 8 * q + 4);
      uint4 v;
      v.x = relu_pack_bf16x2(__uint_as_float(r[8 * q + 0]) + b0.x, __uint_as_float(r[8 * q + 1]) + b0.y);
      v.y = relu_pack_bf16x2(__uint_as_float(r[8 * q + 2]) + b0.z, __uint_as_float(r[8 * q + 3]) + b0.w);
      v.z = relu_pack_bf16x2(__uint_as_float(r[8 * q + 4]) + b1.x, __uint_as_float(r[8 * q + 5]) + b1.y);
      v.w = relu_pack_bf16x2(__uint_as_float(r[8 * q + 6]) + b1.z, __uint_as_float(r[8 * q + 7]) + b1.w);
      *reinterpret_cast<uint4*>(sH + chunk_off(row, (uint32_t)(c0 >> 3) + q, 128)) = v;
    }
  }
}

__global__ void __launch_bounds__(kThreads, 1) actor_forward_kernel(const Args a) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t bars[kSlots];
  __shared__ uint32_t tmem_slot;
  const uint32_t tid = threadIdx.x;
  const int slot = (int)(tid / kSlotThreads);
  const uint32_t row = tid % kSlotThreads, swarp = row >> 5;  // tile row of this thread, warp within the slot
  const int obs_dim = a.p.obs_dim, act_dim = a.p.act_dim;

  // ---- one-time: weights, biases, normalisation constants -> smem; TMEM; barriers
  stage_weight(smem + kSmW1, (const __nv_bfloat16*)a.p.w1, kHid, kIn, tid, kThreads);
  stage_weight(smem + kSmW2, (const __nv_bfloat16*)a.p.w2, kHid, kHid, tid, kThreads);
  stage_weight(smem + kSmWmu, (const __nv_bfloat16*)a.p.w_mu, kHead, kHid, tid, kThreads);
  float* sB1 = reinterpret_cast<float*>(smem + kSmB1);
  float* sB2 = reinterpret_cast<float*>(smem + kSmB2);
  float* sBmu = reinterpret_cast<float*>(smem + kSmBmu);
  float* sMean = reinterpret_cast<float*>(smem + kSmNorm);
  float* sInv = sMean + kIn;
  if (tid < kHid) { sB1[tid] = __ldg(a.p.b1 + tid); sB2[tid] = __ldg(a.p.b2 + tid); }
  if (tid < kHead) sBmu[tid] = __ldg(a.p.b_mu + tid);
  if (tid < kIn) {
    sMean[tid] = (a.obs_mean && (int)tid < obs_dim) ? __ldg(a.obs_mean + tid) : 0.f;
    sInv[tid] = (a.obs_inv_std && (int)tid < obs_dim) ? __ldg(a.obs_inv_std + tid) : 1.f;
  }
  if (tid < 32) tmem_alloc(&tmem_slot, kTmemCols);
  if (tid == 0) {
    for (int s = 0; s < kSlots; ++s) mbar_init(&bars[s], 1);
    mbar_fence_init();
  }
  fence_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();

  uint64_t* bar = &bars[slot];
  const uint32_t tacc = tmem_slot + slot * kSlotTmem;             // MMA destination (lane field 0)
  const uint32_t tacc_row = tacc + ((swarp * 32u) << 16);         // this warp's lane quarter
  uint8_t* slotp = smem + kSmSlot + slot * kSlotBytes;
  const uint32_t sX = smem_u32(slotp + kSlotX), sH = smem_u32(slotp + kSlotH);
  const uint32_t sW1 = smem_u32(smem + kSmW1), sW2 = smem_u32(smem + kSmW2), sWmu = smem_u32(smem + kSmWmu);
  constexpr uint32_t LBO_ACT = 128 * 16, LBO_W1 = kHid * 16, LBO_W2 = kHid * 16, LBO_WMU = kHead * 16;
  const uint32_t idesc_h = make_idesc_bf16(128, kHid), idesc_o = make_idesc_bf16(128, kHead);
  const int64_t n_rows = a.n;
  const int n_tiles = (int)((n_rows + 127) / 128);
  const float clipv = (a.obs_mean && a.obs_clip > 0.f) ? a.obs_clip : 3.0e38f;  // VecNormalize clips what it normalises
  const int tile_stride = a.grid * kSlots, tile0 = slot_major_first_tile(slot, (int)blockIdx.x, a.grid);
  uint32_t phase = 0;

  auto load_x = [&](int tile, float (&x)[kIn]) {
    const int64_t r = (int64_t)tile * 128 + row;
    if (tile >= n_tiles || r >= n_rows) {
#pragma unroll
      for (int j = 0; j < kIn; ++j) x[j] = 0.f;
      return;
    }
    load_f32_row(a.obs + r * a.obs_stride, obs_dim, a.obs_vec != 0, x);
  };
  // VecNormalize.normalize_obs of this thread's row -> bf16 X operand (interleaved K-major) and, if asked, fp32 obs_norm_out
  auto stage_x = [&](int tile, const float (&xraw)[kIn]) {
    const int64_t r = (int64_t)tile * 128 + row;
    const bool valid = r < n_rows;
    float* dst = (a.obs_norm_out && valid) ? a.obs_norm_out + r * obs_dim : nullptr;
#pragma unroll
    for (int q = 0; q < kIn / 8; ++q) {
      float x[8];
      uint32_t w[4];
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const int c = 8 * q + 2 * h;
        x[2 * h] = fminf(fmaxf((xraw[c] - sMean[c]) * sInv[c], -clipv), clipv);
        x[2 * h + 1] = fminf(fmaxf((xraw[c + 1] - sMean[c + 1]) * sInv[c + 1], -clipv), clipv);
        __nv_bfloat162 pk = __floats2bfloat162_rn(x[2 * h], x[2 * h + 1]);
        w[h] = *reinterpret_cast<uint32_t*>(&pk);
      }
      *reinterpret_cast<uint4*>(slotp + kSlotX + chunk_off(row, q, 128)) = make_uint4(w[0], w[1], w[2], w[3]);
      if (dst && 8 * q < obs_dim) {
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int c0 = 8 * q + 4 * v;
          if (a.norm_vec && c0 + 4 <= obs_dim) {
            *reinterpret_cast<float4*>(dst + c0) = make_float4(x[4 * v], x[4 * v + 1], x[4 * v + 2], x[4 * v + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (c0 + j < obs_dim) dst[c0 + j] = x[4 * v + j];
          }
        }
      }
    }
  };
  auto issue_l1 = [&]() {
#pragma unroll
    for (int ks = 0; ks < kIn / 16; ++ks)
      mma_bf16(tacc, make_desc(sX + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW1 + ks * 2 * LBO_W1, LBO_W1, 128), idesc_h, ks > 0);
  };

  if (tile0 < n_tiles) {
    float xbuf[kIn];
    load_x(tile0, xbuf);
    stage_x(tile0, xbuf);
    load_x(tile0 + tile_stride, xbuf);
    fence_async_smem();
    fence_before_sync();
    slot_barrier(slot, kSlotThreads);
    if (row == 0) { fence_after_sync(); issue_l1(); mma_commit(bar); }
    for (int tile = tile0; tile < n_tiles; tile += tile_stride) {
      const int next = tile + tile_stride;
      // ---- L1 done: X is free -- stage the next tile (raw rows in xbuf) and request the one after
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      if (next < n_tiles) {
        stage_x(next, xbuf);
        load_x(next + tile_stride, xbuf);
      }
      relu_epilogue(tacc_row, sB1, slotp + kSlotH, row);
      fence_async_smem();
      fence_before_sync();
      slot_barrier(slot, kSlotThreads);
      // ---- L2
      if (row == 0) {
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < kHid / 16; ++ks)
          mma_bf16(tacc, make_desc(sH + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sW2 + ks * 2 * LBO_W2, LBO_W2, 128), idesc_h, ks > 0);
        mma_commit(bar);
      }
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      relu_epilogue(tacc_row, sB2, slotp + kSlotH, row);
      fence_async_smem();
      fence_before_sync();
      slot_barrier(slot, kSlotThreads);
      // ---- L3: action head into accumulator columns 0..15
      if (row == 0) {
        fence_after_sync();
#pragma unroll
        for (int ks = 0; ks < kHid / 16; ++ks)
          mma_bf16(tacc, make_desc(sH + ks * 2 * LBO_ACT, LBO_ACT, 128), make_desc(sWmu + ks * 2 * LBO_WMU, LBO_WMU, 128), idesc_o, ks > 0);
        mma_commit(bar);
      }
      mbar_wait(bar, phase); phase ^= 1;
      fence_after_sync();
      {
        uint32_t r[16];
        tmem_ld16(tacc_row, r);
        tmem_ld_wait();
        const int64_t grow = (int64_t)tile * 128 + row;
        if (grow < n_rows) {
          float act[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < act_dim) act[j] = accurate_tanh(__uint_as_float(r[j]) + sBmu[j]);  // SquashedDiagGaussian mode
          if (a.act_vec) {
            *reinterpret_cast<float4*>(a.actions + grow * 4) = make_float4(act[0], act[1], act[2], act[3]);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < act_dim) a.actions[grow * act_dim + j] = act[j];
          }
        }
      }
      // every thread has read the head columns before the next L1 overwrites them
      fence_before_sync();
      slot_barrier(slot, kSlotThreads);
      if (row == 0 && next < n_tiles) { fence_after_sync(); issue_l1(); mma_commit(bar); }
    }
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  if (tid < 32) tmem_dealloc(tmem_slot, kTmemCols);
}

}  // namespace sac

static bool aligned(const void* p, uintptr_t bytes) { return ((uintptr_t)p & (bytes - 1)) == 0; }

static bool actor_ok(const SacActor* p) {
  return p && p->w1 && p->w2 && p->w_mu && p->b1 && p->b2 && p->b_mu && aligned(p->w1, 16) && aligned(p->w2, 16) && aligned(p->w_mu, 16) &&
         aligned(p->b1, 4) && aligned(p->b2, 4) && aligned(p->b_mu, 4) && p->obs_dim >= 1 && p->obs_dim <= SAC_IN_PAD && p->act_dim >= 1 &&
         p->act_dim <= 4;
}

extern "C" int sac_actor_forward(const SacActor* actor, const float* obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                                 const float* obs_inv_std, float obs_clip, float* actions, float* obs_norm_out, void* stream) {
  if (!actor_ok(actor) || !obs || !aligned(obs, 4) || n <= 0 || n > (int64_t)INT_MAX * 64 || obs_stride < actor->obs_dim || !actions ||
      !aligned(actions, 4) || !aligned(obs_norm_out, 4) || (!obs_mean) != (!obs_inv_std) || !aligned(obs_mean, 4) || !aligned(obs_inv_std, 4))
    return qx_fail(QX_EINVAL, "%s", "sac_actor_forward: bad arguments");
  sac::Args a{};
  a.p = *actor; a.obs = obs; a.obs_stride = obs_stride; a.n = n; a.obs_mean = obs_mean; a.obs_inv_std = obs_inv_std; a.obs_clip = obs_clip;
  a.actions = actions; a.obs_norm_out = obs_norm_out;
  a.obs_vec = aligned(obs, 16) && (obs_stride & 3) == 0;
  a.norm_vec = (actor->obs_dim & 3) == 0 && aligned(obs_norm_out, 16);
  a.act_vec = actor->act_dim == 4 && aligned(actions, 16);
  // per device: SM count and the one-time opt-in to ~205 KB of dynamic shared memory (cached only after the call succeeded)
  static std::atomic<int> sms_of[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return qx_fail(QX_ECUDA, "%s", "sac_actor_forward: cannot query the current device");
  int sms = sms_of[dev].load(std::memory_order_acquire);
  if (!sms) {
    int m = 0;
    if (cudaDeviceGetAttribute(&m, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || m <= 0)
      return qx_fail(QX_ECUDA, "%s", "sac_actor_forward: cannot query the SM count");
    if (cudaFuncSetAttribute(sac::actor_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sac::kSmTotal) != cudaSuccess)
      return qx_fail(QX_ECUDA, "%s", "sac_actor_forward: cannot reserve shared memory");
    sms_of[dev].store(m, std::memory_order_release);
    sms = m;
  }
  const int64_t tiles = (n + 127) / 128;
  const unsigned grid = (unsigned)(tiles < sms ? tiles : sms);  // small batches: one tile per SM before a second slot is used
  a.grid = (int32_t)grid;
  sac::actor_forward_kernel<<<grid, sac::kThreads, sac::kSmTotal, (cudaStream_t)stream>>>(a);
  return cudaGetLastError() == cudaSuccess ? QX_OK : qx_fail(QX_ECUDA, "%s", "sac_actor_forward: launch failed");
}
