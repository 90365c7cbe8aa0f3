// qx_kernels.cu -- K1: the fused env-step kernel (one thread per env) and the
// C-ABI of include/quadx_b200.h.  sm_100a only.
//
// One launch of quadx_step_kernel does, per env, what the reference does in
// QuadXHoverEnv.step (hover.py:334-358): scale the action, run 6 Aviary.step()
// = 12 physics sub-steps with the rate PID every 2nd, build the 20-D
// observation, compute reward / termination / truncation, and -- with
// auto_reset -- the whole of reset() (hover.py:72-113, incl. its 10 idle
// Aviary.step()) for the envs that finished.  The 44 carried words are read
// once as 11 coalesced float4 loads, live in registers across the sub-steps,
// and are written back once.
#include <cooperative_groups.h>
#include <cooperative_groups/reduce.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <new>

#include "../../include/quadx_b200.h"
#include "qx_internal.h"
#include "qx_model.cuh"

namespace qx {

#ifndef QX_BLOCK
#define QX_BLOCK 128
#endif
#ifndef QX_MIN_BLOCKS
#define QX_MIN_BLOCKS 4
#endif
#ifndef QX_PAIR_UNROLL
#define QX_PAIR_UNROLL 1
#endif
constexpr int kBlock = QX_BLOCK;

struct Stats {
  double sum_ret;
  unsigned long long sum_len;
  unsigned long long n_done;
  unsigned long long n_nonfinite;  // envs whose state stopped being finite and were terminated (failure detection)
};

// Envs that finished in a step and must be re-created before the next one.
// Filled by the step kernel, drained by the reset kernel launched right after
// it on the same stream, so that reset work (20 idle sub-steps, hover.py:109)
// runs in full warps instead of diverging inside the step kernel.
struct ResetQueue {
  unsigned int count;
  unsigned int ticket;
  // merged step kernel (quadx_step_hot_kernel<..., MERGED>): block tickets of one launch, re-armed by the last block to
  // leave, and the number of envs the launch queued (count itself is zero again when the launch ends)
  unsigned int tasks_done, next_reset, exit_ticket, published;
  unsigned int pad[2];
  unsigned int idx[1];  // [n_envs]
};

struct StepArgs {
  float4* state;
  const float* actions;     // [k, n, act_dim]
  void* obs;                // [k, n, obs_stride]
  float* reward;            // [k, n]
  uint8_t* terminated;      // [k, n]
  uint8_t* truncated;       // [k, n]
  float* terminal_obs;      // [n, obs_dim] or null
  const uint8_t* mask;      // reset only
  Stats* stats;
  ResetQueue* queue;        // deferred-reset mode (MODE_STEP_DEFER / MODE_RESET_QUEUE)
  int64_t n;
  int64_t env_begin, env_count;  // step modes: the env sub-range this launch covers (host-side chunked pipeline)
  int64_t obs_stride;
  int32_t k;
  int32_t obs_bf16;
  int32_t stream_stores;    // hot kernel: 1 = observations / reward / flags with evict-first stores (write-once data), 2 = the state planes too
  int32_t merged;           // hot kernel: the last resident wave of blocks drains the reset queue in the same launch
  uint32_t drainers;        // ... and this is how many blocks that wave has (resident blocks per SM x SMs)
  int32_t paired_reset;     // queued envs are re-created by the paired code (hot_reset_env): even idle sub-step count, throttles >= 0
};

template <int DIM>
__device__ __forceinline__ void write_obs(const float (&o)[DIM], void* base, int64_t row, int64_t stride, bool bf16, bool cs = false) {
  static_assert(DIM % 4 == 0, "obs rows are written as 16-byte / 8-byte vectors");
  if (bf16) {
    __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(base) + row * stride;
    if ((stride & 3) == 0) {
#pragma unroll
      for (int j = 0; j < DIM; j += 4) {
        __nv_bfloat162 a = __floats2bfloat162_rn(o[j], o[j + 1]), b = __floats2bfloat162_rn(o[j + 2], o[j + 3]);
        uint2 v;
        v.x = *reinterpret_cast<uint32_t*>(&a);
        v.y = *reinterpret_cast<uint32_t*>(&b);
        if (cs) __stcs(reinterpret_cast<uint2*>(p + j), v);
        else *reinterpret_cast<uint2*>(p + j) = v;
      }
    } else {
#pragma unroll
      for (int j = 0; j < DIM; ++j) p[j] = __float2bfloat16_rn(o[j]);
    }
  } else {
    float* p = reinterpret_cast<float*>(base) + row * stride;
    if ((stride & 3) == 0) {
#pragma unroll
      for (int j = 0; j < DIM; j += 4) {
        if (cs) __stcs(reinterpret_cast<float4*>(p + j), make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]));
        else *reinterpret_cast<float4*>(p + j) = make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < DIM; ++j) p[j] = o[j];
    }
  }
}

// MODE_STEP_INLINE : k agent steps, finished envs reset inside the same thread (qx_step_k)
// MODE_STEP_DEFER  : one agent step, finished envs are queued for MODE_RESET_QUEUE (qx_step)
// MODE_RESET_MASK  : qx_reset (masked reset, no step)
// MODE_RESET_QUEUE : reset of the envs queued by the preceding MODE_STEP_DEFER launch
enum { MODE_STEP_INLINE = 0, MODE_STEP_DEFER = 1, MODE_RESET_MASK = 2, MODE_RESET_QUEUE = 3 };

// CASC: the instantiation for PyFlyt flight modes != 0 (outer PID loops; 6 more state planes).  hover.py itself only
// ever reaches mode 0 (set_mode(0), hover.py:92), which is the CASC = false path.
template <int MODE, int TASK, bool CASC, bool NC = true>
__device__ __forceinline__ void run_env(const DevConfig& c, const StepArgs& a, int64_t i);

constexpr int kResetQueueBlocks = 148 * 4;  // persistent grid of the queue-draining launch

// Deferred-reset step launches: the last block to finish copies the queue length to ResetQueue.published, which is what
// qx_done_queue hands out -- it stays valid while the reset launch (which zeroes count) runs, so a consumer of the queue
// (the rollout's time-limit bootstrap) may run concurrently with the reset.  No fence: every count atomic of a block has
// returned (its result was used) before the block's __syncthreads, and atomics are performed at L2.
__device__ __forceinline__ void publish_queue_length(ResetQueue* q) {
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(&q->tasks_done, 1u) == gridDim.x - 1) {
      q->published = atomicAdd(&q->count, 0u);
      q->tasks_done = 0u;
    }
  }
}

// REF: the model constants are the reference's literals (qx_ref_constants.cuh) instead of kernel parameters
template <int MODE, int TASK, bool CASC = false, bool REF = false>
__global__ void __launch_bounds__(kBlock, QX_MIN_BLOCKS) quadx_step_kernel(const __grid_constant__ DevConfig cparam, const __grid_constant__ StepArgs a) {
  if (MODE == MODE_STEP_INLINE) {
    // launched as a programmatic dependent of whatever kernel precedes it on the stream (launch_task): wait for that grid and its
    // memory, then let the next launch of the chain be scheduled while this one runs (small batches are launch-latency-bound)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
  }
  DevConfig cref = cparam;  // scalar-replaced by the compiler: untouched fields stay parameter reads
  if (REF) apply_ref_constants(cref);
  const DevConfig& c = REF ? cref : cparam;
  if (MODE == MODE_RESET_QUEUE) {
    // Every block reads the count before any block can zero it: the zeroing
    // block is the last one to take a ticket, after its own __syncthreads.
    const unsigned int cnt = *reinterpret_cast<volatile unsigned int*>(&a.queue->count);
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(&a.queue->ticket, 1u) == gridDim.x - 1) { a.queue->count = 0u; a.queue->ticket = 0u; }
    }
    for (unsigned int t = blockIdx.x * kBlock + threadIdx.x; t < cnt; t += gridDim.x * kBlock)
      run_env<MODE, TASK, CASC>(c, a, (int64_t)a.queue->idx[t]);
  } else if (MODE == MODE_STEP_DEFER) {
    const int64_t i = a.env_begin + (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i < a.env_begin + a.env_count) run_env<MODE, TASK, CASC>(c, a, i);
    publish_queue_length(a.queue);
  } else {
    const int64_t i = a.env_begin + (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= a.env_begin + a.env_count) return;
    if (MODE == MODE_RESET_MASK && a.mask && !a.mask[i]) return;
    run_env<MODE, TASK, CASC>(c, a, i);
  }
}

// cascade only: what Aviary.reset() + QuadX.set_mode(mode) leave behind -- cleared outer-loop memory, the Euler row
// of the fresh snapshot, and set_mode's preset setpoint (hold the current height in modes 2-4, the pose in mode 7)
__device__ __forceinline__ void respawn_cascade(Env& e, const DevConfig& c, float seul[3], float sp[4]) {
#pragma unroll
  for (int k = 0; k < 18; ++k) e.cp[k] = 0.f;
  quat_to_euler(e.sqx, e.sqy, e.sqz, e.sqw, seul[0], seul[1], seul[2]);
  sp[0] = sp[1] = sp[2] = sp[3] = 0.f;
  if (c.flight_mode == 2 || c.flight_mode == 3 || c.flight_mode == 4) sp[3] = e.spz;
  if (c.flight_mode == 7) { sp[0] = e.spx; sp[1] = e.spy; sp[2] = seul[2]; sp[3] = e.spz; }
}

template <int TASK> struct ObsDim { static constexpr int value = TASK == QX_TASK_HOVER ? QX_OBS_DIM_HOVER : QX_OBS_DIM_YAW; };
struct ObsAux { float er, ep, ey, cx, cy, area, ratio; bool vis; };

// ---- compute_attitude / compute_state, hover.py:224-272 (phase 0: after an agent step, 1: first observation of an episode)
// RASTER_OK: the instantiation may take the vision_mode = 1 branch (a non-inlined call; the lean hot kernels leave it out --
// a handle in that mode runs the generic kernels -- so that the call's ABI does not cost their sub-step loop registers)
template <int TASK, bool RASTER_OK = true>
__device__ __forceinline__ void build_obs(Env& e, const DevConfig& c, const float act[4], const int phase, const bool live,
                                          float (&obs)[ObsDim<TASK>::value], ObsAux& x) {
  float er, ep, ey;
  if (phase == 0 && !live) {
    er = e.peul[0]; ep = e.peul[1]; ey = e.peul[2];  // frozen after the episode ended
  } else {
    quat_to_euler(e.sqx, e.sqy, e.sqz, e.sqw, er, ep, ey);
  }
  if (phase == 1) { e.peul[0] = er; e.peul[1] = ep; e.peul[2] = ey; }  // hover.py:112
  const float two_pi = 6.28318530718f, pi = 3.14159265359f;
  float d0 = er - e.peul[0] + pi, d1 = ep - e.peul[1] + pi, d2 = ey - e.peul[2] + pi;
  d0 = d0 - two_pi * floorf(d0 * (1.f / two_pi)) - pi;  // hover.py:229 (python floor-mod)
  d1 = d1 - two_pi * floorf(d1 * (1.f / two_pi)) - pi;
  d2 = d2 - two_pi * floorf(d2 * (1.f / two_pi)) - pi;
  bool vis;
  float cx, cy, area = 0.f, ratio = 0.f;
  if (TASK == QX_TASK_HOVER) {
    if (RASTER_OK && c.vision_mode == 1) vision_raster(e.px, e.py, e.pz, e.qx, e.qy, e.qz, e.qw, c.raster, vis, cx, cy, area, ratio);
    else vision(e, c, vis, cx, cy, area, ratio);
    obs[0] = d0 * c.inv_agent_dt; obs[1] = d1 * c.inv_agent_dt; obs[2] = d2 * c.inv_agent_dt;
    euler_to_quat(er, ep, ey, obs[3], obs[4], obs[5], obs[6]);  // hover.py:233
    obs[7] = cx; obs[8] = cy; obs[9] = e.pcx; obs[10] = e.pcy;
    obs[11] = area; obs[12] = e.parea; obs[13] = vis ? 1.f : 0.f; obs[14] = ratio; obs[15] = e.pratio;
    obs[16] = act[0]; obs[17] = act[1]; obs[18] = act[2]; obs[19] = act[3];
    e.pcx = cx; e.pcy = cy; e.parea = area; e.pratio = ratio;  // hover.py:270-272
  } else {
    // yaw.py:57-74: [euler / pi (3) | sphere centre (2) | angular velocity (3) | last 4 yaw actions (4)].  The
    // reference's sphere detector and calculate_angular_velocity are missing; declared stand-ins: the analytic
    // projection of the sphere centre, and the wrapped Euler finite difference of hover.py:228-230 scaled by the
    // 30 rad/s command range into the Box(-1, 1) of yaw.py:41-45.
    vision_point(e, c, vis, cx, cy);
    const float k = c.inv_agent_dt * (1.f / 30.f);
    obs[0] = er * (1.f / pi); obs[1] = ep * (1.f / pi); obs[2] = ey * (1.f / pi);
    obs[3] = cx; obs[4] = cy;
    obs[5] = clampf(d0 * k, -1.f, 1.f); obs[6] = clampf(d1 * k, -1.f, 1.f); obs[7] = clampf(d2 * k, -1.f, 1.f);
    obs[8] = e.pa[0]; obs[9] = e.pa[1]; obs[10] = e.pa[2]; obs[11] = e.pa[3];
    e.pcx = cx; e.pcy = cy;
  }
  x.er = er; x.ep = ep; x.ey = ey; x.cx = cx; x.cy = cy; x.area = area; x.ratio = ratio; x.vis = vis;
}

// ---- compute_term_trunc_reward (hover.py:274-332) / yaw.py:138-149 + the end-of-step bookkeeping (hover.py:354-357).
// Writes reward and flags of this step; returns true when the episode ended and the env must be re-created.
template <int TASK, bool CASC>
__device__ __forceinline__ bool reward_and_flags(Env& e, const DevConfig& c, const StepArgs& a, const int64_t row, const float act[4],
                                                 const bool live, float (&obs)[ObsDim<TASK>::value], const ObsAux& x) {
  constexpr int OBS_DIM = ObsDim<TASK>::value;
  if (TASK == QX_TASK_YAW) {
    // calculate_reward is missing from the reference; declared stand-in:
    // keep the sphere horizontally centred, 1 - |cx| when seen else -1, minus 0.05 |a_t - a_(t-1)|.
    uint32_t fl = e.flags;
    if (e.step_count >= c.max_steps) fl |= F_TRUNC;  // yaw.py:138-139
    if (e.spx * e.spx + e.spy * e.spy + e.spz * e.spz > c.dome2) fl |= F_OOB | F_TERM;  // yaw.py:141-143
    const float reward = (x.vis ? 1.f - fabsf(x.cx) : -1.f) - 0.05f * fabsf(e.pa[3] - e.pa[2]);
    e.flags = fl;
    e.peul[0] = x.er; e.peul[1] = x.ep; e.peul[2] = x.ey;
    e.step_count += 1;  // yaw.py:145
    e.rng_ctr += 1u;
    e.ep_ret += reward;
    a.reward[row] = reward;
    a.terminated[row] = (fl & F_TERM) ? 1 : 0;
    a.truncated[row] = (fl & F_TRUNC) ? 1 : 0;
    return c.auto_reset && (fl & (F_TERM | F_TRUNC));
  }
  float reward = -0.1f;  // hover.py:343
  uint32_t fl = e.flags;
  if (e.step_count > c.max_steps) fl |= F_TRUNC;  // hover.py:275-276
  if (live) {
    fl &= ~(F_LOWZ);
    if (e.spx * e.spx + e.spy * e.spy + e.spz * e.spz > c.dome2) fl |= F_OOB;
    if (e.spz < c.floor_thr) fl |= F_LOWZ;
  }
  bool bad = false;
  // failure containment (no counterpart in the reference): a state that is no longer finite ends the episode like
  // an out-of-bounds flight, is counted, and the env is re-created by the auto-reset -- it cannot poison the batch
  if (live && !(fabsf(e.px) + fabsf(e.py) + fabsf(e.pz) + fabsf(e.vx) + fabsf(e.vy) + fabsf(e.vz) + fabsf(e.wx) + fabsf(e.wy) + fabsf(e.wz) +
                fabsf(e.qw) < 3.0e38f)) {
    fl |= F_OOB;
    bad = true;
    atomicAdd(&a.stats->n_nonfinite, 1ull);
    e.px = e.py = 0.f; e.pz = c.floor_z; e.vx = e.vy = e.vz = 0.f; e.wx = e.wy = e.wz = 0.f; e.qx = e.qy = e.qz = 0.f; e.qw = 1.f;
#pragma unroll
    for (int m = 0; m < 4; ++m) e.thr[m] = 0.f;
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) { e.pi[ax] = e.pe[ax] = e.swb[ax] = e.svb[ax] = 0.f; }
    if (CASC) {
#pragma unroll
      for (int k = 0; k < 18; ++k) e.cp[k] = 0.f;
      e.spx = e.spy = 0.f; e.spz = c.floor_z;
    }
  }
  if (fl & F_OOB) { reward = -100.f; fl |= F_TERM; }  // hover.py:278-281
  if (e.step_count > c.floor_grace && !c.render && (fl & F_LOWZ)) {  // hover.py:283-290
    reward = -100.f; fl |= F_TERM | F_ONFLOOR;
  }
  const float target_reward =
      x.vis ? -(fsqrt(x.cx * x.cx + x.cy * x.cy) + fabsf(x.area - c.target_area) + fabsf(x.ratio - c.target_ratio)) : -2.0f;
  reward -= 0.01f * e.swb[2] * e.swb[2];                        // hover.py:322-324
  reward += target_reward - fsqrt(x.er * x.er + x.ep * x.ep);  // hover.py:326-327
  const float a0 = act[0] - e.pa[0], a1 = act[1] - e.pa[1], a2 = act[2] - e.pa[2], a3 = act[3] - e.pa[3];
  reward -= 0.2f * fsqrt(a0 * a0 + a1 * a1 + a2 * a2 + a3 * a3);  // hover.py:329-331
  reward += 1.0f;                                               // hover.py:332
  if (bad) {  // nothing derived from the broken state may leave the kernel
    reward = -100.f;
#pragma unroll
    for (int j = 0; j < OBS_DIM; ++j) obs[j] = 0.f;
  }
  e.flags = fl;
  e.peul[0] = x.er; e.peul[1] = x.ep; e.peul[2] = x.ey;  // hover.py:354
  e.step_count += 1;                                     // hover.py:356
  e.pa[0] = act[0]; e.pa[1] = act[1]; e.pa[2] = act[2]; e.pa[3] = act[3];  // hover.py:357
  e.rng_ctr += 1u;
  e.ep_ret += reward;
  const bool term = fl & F_TERM, trunc = fl & F_TRUNC;
  if (a.stream_stores) {  // write-once results: evict-first, so that they do not displace the state planes in L2
    __stcs(a.reward + row, reward);
    __stcs(a.terminated + row, (uint8_t)(term ? 1 : 0));
    __stcs(a.truncated + row, (uint8_t)(trunc ? 1 : 0));
  } else {
    a.reward[row] = reward;
    a.terminated[row] = term ? 1 : 0;
    a.truncated[row] = trunc ? 1 : 0;
  }
  return c.auto_reset && (term || trunc);
}

// ---- SB3 VecEnv auto-reset + Monitor episode statistics.  The lanes of the warp that finished together aggregate: one
// atomic per counter per warp (a mass termination -- e.g. every env hitting the floor rule on its 32nd step -- would
// otherwise serialise ~4 atomics per env on four L2 addresses).  DEFER: the env is handed to the reset kernel, which
// writes the next observation.
template <bool DEFER, int OBS_DIM>
__device__ __forceinline__ void episode_end(const Env& e, const StepArgs& a, const int64_t i, const float (&obs)[OBS_DIM]) {
  namespace cg = cooperative_groups;
  const auto g = cg::coalesced_threads();
  const double sr = cg::reduce(g, (double)e.ep_ret, cg::plus<double>());
  const unsigned long long sl = cg::reduce(g, (unsigned long long)e.step_count, cg::plus<unsigned long long>());
  unsigned int base = 0;
  if (g.thread_rank() == 0) {
    atomicAdd(&a.stats->sum_ret, sr);
    atomicAdd(&a.stats->sum_len, sl);
    atomicAdd(&a.stats->n_done, (unsigned long long)g.size());
    if (DEFER) base = atomicAdd(&a.queue->count, (unsigned int)g.size());
  }
  if (a.terminal_obs) write_obs(obs, a.terminal_obs, i, OBS_DIM, false);
  if (DEFER) {
    base = g.shfl(base, 0);
    a.queue->idx[base + g.thread_rank()] = (unsigned int)i;
  }
}

template <int MODE, int TASK, bool CASC, bool NC>
__device__ __forceinline__ void run_env(const DevConfig& c, const StepArgs& a, const int64_t i) {
  constexpr int OBS_DIM = ObsDim<TASK>::value;
  constexpr bool RESET_ONLY = MODE == MODE_RESET_MASK || MODE == MODE_RESET_QUEUE;
  Env e;
  load_env<NC>(e, a.state, a.n, i);
  if (CASC) load_cascade(e, a.state, a.n, i);
  float seul[3];  // cascade: Euler row of the Aviary.state snapshot
  const uint32_t k0 = c.seed_lo ^ (c.env_lo + (uint32_t)i);
  const uint32_t k1 = c.seed_hi ^ (c.env_hi + (uint32_t)(((uint64_t)c.env_lo + (uint64_t)i) >> 32));

  for (int kk = 0; kk < ((RESET_ONLY || MODE == MODE_STEP_DEFER) ? 1 : a.k); ++kk) {
    const int64_t row = (int64_t)kk * a.n + i;
    float act[4] = {0.f, 0.f, 0.f, 0.f};
    float sp[4] = {0.f, 0.f, 0.f, 0.f};
    seul[0] = e.peul[0]; seul[1] = e.peul[1]; seul[2] = e.peul[2];  // == previous_ang_pos (hover.py:112,354) between steps
    int phase = RESET_ONLY ? 1 : 0;  // 0: the agent step, 1: reset (idle steps + first obs)
    int nsub;
    if (RESET_ONLY) {
      respawn(e, c, k0, k1);
      if (CASC) respawn_cascade(e, c, seul, sp);
      nsub = c.n_sub_reset;
    } else {
      if (TASK == QX_TASK_HOVER) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(a.actions) + row);
        act[0] = v.x; act[1] = v.y; act[2] = v.z; act[3] = v.w;
        sp[0] = act[0] * c.act_scale[0];  // hover.py:337-341
        sp[1] = act[1] * c.act_scale[1];
        sp[2] = act[2] * c.act_scale[2];
        sp[3] = fmaf(act[3], c.thrust_scale, c.thrust_bias);
        if (!CASC) sp[3] = __saturatef(sp[3]);  // QuadX.update_control clips the mode-0 thrust command to [0, 1]
        if (CASC && c.flight_mode == -1) {      // four motor pwm commands: all of them through the throttle mapping
#pragma unroll
          for (int m = 0; m < 3; ++m) sp[m] = fmaf(act[m], c.thrust_scale, c.thrust_bias);
        }
      } else {
        act[0] = __ldg(a.actions + row);  // yaw.py:105-122: roll = pitch = 0, yaw * -30, throttle (-1 + 1) / 2 = 0
        sp[2] = act[0] * c.act_scale[2];
        e.pa[0] = e.pa[1]; e.pa[1] = e.pa[2]; e.pa[2] = e.pa[3]; e.pa[3] = act[0];  // yaw.py:108 action_history.append
      }
      nsub = (TASK == QX_TASK_HOVER && (e.flags & (F_TERM | F_TRUNC))) ? 0 : c.n_sub_step;  // hover.py:347-348; yaw.py:126 always steps
    }
    const bool live = RESET_ONLY || nsub > 0 || c.n_sub_step == 0;
    float obs[OBS_DIM];
    bool deferred = false;

    while (true) {
      // ---- Aviary.step() x ratio: control on every ctrl_every-th sub-step
      float pwm[4] = {0.f, 0.f, 0.f, 0.f};
      const uint32_t stream = phase ? STREAM_RESET : STREAM_STEP;
#ifndef QX_NO_PAIR_LOOP
      constexpr bool kPairLoop = true;
#else
      constexpr bool kPairLoop = false;
#endif
      if (kPairLoop && c.ctrl_every == 2 && (nsub & 1) == 0) {
        // default scheduling (control_hz = physics_hz / 2): one rate-PID update and one Philox call per
        // Aviary.step(), then its two physics sub-steps
        constexpr int kPairUnroll = QX_PAIR_UNROLL;
#pragma unroll kPairUnroll
        for (int j = 0; j < nsub; j += 2) {
          if (CASC) control_update_cascade(e, c, sp, seul, pwm);
          else control_update<float>(e, c, sp, pwm);
          float nz[4] = {0.f, 0.f, 0.f, 0.f};
          uint4 bits = make_uint4(0u, 0u, 0u, 0u);
          if (c.noise) {
            bits = env_philox(make_uint4((uint32_t)j >> 1, stream, e.rng_ctr, 0u), k0, k1);
            normal4_scaled<float>(bits.x, bits.y, c.noise_k, nz);
          }
          physics_substep<float>(e, c, pwm, nz, false);
          if (c.noise) normal4_scaled<float>(bits.z, bits.w, c.noise_k, nz);
          physics_substep<float>(e, c, pwm, nz, CASC || j + 2 == nsub);  // the outer loops read the snapshot pose at every control update
          if (CASC && c.need_euler) quat_to_euler(e.sqx, e.sqy, e.sqz, e.sqw, seul[0], seul[1], seul[2]);
        }
      } else {
        uint4 bits = make_uint4(0u, 0u, 0u, 0u);
        for (int j = 0, cc = 0; j < nsub; ++j) {
          if (cc == 0) {
            if (CASC) {
              if (j > 0 && c.need_euler) quat_to_euler(e.sqx, e.sqy, e.sqz, e.sqw, seul[0], seul[1], seul[2]);
              control_update_cascade(e, c, sp, seul, pwm);
            } else {
              control_update<float>(e, c, sp, pwm);
            }
          }
          if (++cc == c.ctrl_every) cc = 0;
          float nz[4] = {0.f, 0.f, 0.f, 0.f};
          if (c.noise) {  // one Philox call feeds two sub-steps
            if ((j & 1) == 0) bits = env_philox(make_uint4((uint32_t)j >> 1, stream, e.rng_ctr, 0u), k0, k1);
            normal4_scaled<float>((j & 1) ? bits.z : bits.x, (j & 1) ? bits.w : bits.y, c.noise_k, nz);
          }
          physics_substep<float>(e, c, pwm, nz, CASC || j + 1 == nsub);
        }
      }
      ObsAux x;
      build_obs<TASK>(e, c, act, phase, live, obs, x);
      if (phase == 1) break;
      if (!reward_and_flags<TASK, CASC>(e, c, a, row, act, live, obs, x)) break;
      episode_end<MODE == MODE_STEP_DEFER>(e, a, i, obs);
      if (MODE == MODE_STEP_DEFER) { deferred = true; break; }
      respawn(e, c, k0, k1);
      act[0] = act[1] = act[2] = act[3] = 0.f;  // hover.py:101
      sp[0] = sp[1] = sp[2] = sp[3] = 0.f;      // set_mode(0): zero setpoint
      if (CASC) respawn_cascade(e, c, seul, sp);
      phase = 1;
      nsub = c.n_sub_reset;
    }
    if (a.obs && !deferred) write_obs(obs, a.obs, RESET_ONLY ? i : row, a.obs_stride, a.obs_bf16 != 0);
  }
  store_env(e, a.state, a.n, i);
  if (CASC) store_cascade(e, a.state, a.n, i);
  if (MODE == MODE_STEP_DEFER && a.merged) __threadfence();  // cold path of the merged launch (see hot_epilogue_loaded)
}

// ===========================================================================
// The two-envs-per-thread step kernel (hover task, flight mode 0, default control scheduling): thread t of a block
// owns envs base + t and base + kPairBlock + t, one in each half of a float2, so the 12 sub-steps run as packed
// FFMA2 / FMUL2 / FADD2 (qx_lanes.cuh).  The once-per-step epilogue (Euler angles, camera, reward, flags) runs per env
// on the scalar code above.  One agent step per launch; finished envs go to the reset queue (auto_reset) like
// MODE_STEP_DEFER.  An env that is already finished on entry (only possible without auto_reset, or when the caller
// skipped qx_step_end) sends its thread through the one-env code instead.
// ===========================================================================
// launch shapes (threads per block, resident blocks per SM -> register cap 65536 / (threads x blocks)).
// QX_SHAPE at qx_create picks one (tuning / profiling); the defaults are the fastest measured on B200.
template <int SHAPE> struct HotShape;
template <> struct HotShape<0> { static constexpr int kBlock = 128, kMinBlocks = 3; };  // 168 registers
template <> struct HotShape<3> { static constexpr int kBlock = 128, kMinBlocks = 4; };  // 128
template <> struct HotShape<4> { static constexpr int kBlock = 128, kMinBlocks = 5; };  // 96
template <> struct HotShape<5> { static constexpr int kBlock = 128, kMinBlocks = 6; };  // 80
#ifdef QX_EXTRA_SHAPES  // tuning builds: small blocks (finer-grained block turnover, 21-23 warps per SM), S1 lanes only
template <> struct HotShape<6> { static constexpr int kBlock = 64, kMinBlocks = 11; };  // 88 registers, 22 warps
template <> struct HotShape<7> { static constexpr int kBlock = 32, kMinBlocks = 23; };  // 88 registers, 23 warps
template <> struct HotShape<8> { static constexpr int kBlock = 64, kMinBlocks = 10; };  // 96 registers, 20 warps
template <> struct HotShape<9> { static constexpr int kBlock = 32, kMinBlocks = 21; };  // 96 registers, 21 warps
constexpr int kHotShapes = 10;
#else
constexpr int kHotShapes = 6;
#endif

template <bool REF>
__device__ __noinline__ void run_env_cold(const DevConfig& cparam, const StepArgs& a, const int64_t i) {
  DevConfig cref = cparam;
  if (REF) apply_ref_constants(cref);
  const DevConfig& c = REF ? cref : cparam;
  if (c.auto_reset) run_env<MODE_STEP_DEFER, QX_TASK_HOVER, false>(c, a, i);
  else run_env<MODE_STEP_INLINE, QX_TASK_HOVER, false>(c, a, i);
}

// one lane of a two-lane value, or the value itself
template <int HALF> QX_DI float half_of(float v) { return v; }
template <int HALF, bool PK> QX_DI float half_of(P2<PK> v) { return HALF ? v.y : v.x; }
template <class V> struct LaneOps;
template <> struct LaneOps<float> {
  static QX_DI float make(float a, float) { return a; }
  static QX_DI void pack(Core<float>& p, const Core<float>& a, const Core<float>&) { p = a; }
};
template <bool PK> struct LaneOps<P2<PK>> {
  static QX_DI P2<PK> make(float a, float b) { return P2<PK>{a, b}; }
  static QX_DI void pack(Core<P2<PK>>& p, const Core<float>& a, const Core<float>& b) { pack_core(p, a, b); }
};
template <int HALF> QX_DI void unpack_lane(Core<float>& a, const Core<float>& p) { a = p; }
template <int HALF, bool PK> QX_DI void unpack_lane(Core<float>& a, const Core<P2<PK>>& p) { unpack_core<HALF>(a, p); }

// once-per-step epilogue of one env of the hot kernel: observation, reward, flags, episode end, state store
template <bool REF>
QX_DI void hot_epilogue_loaded(Env& e, const DevConfig& c, const StepArgs& a, const int64_t i, const float4 av);
template <bool REF>
QX_DI void hot_epilogue(Env& e, const DevConfig& c, const StepArgs& a, const int64_t i, const float4 av) {
  load_env_tail(e, a.state, a.n, i);  // the epilogue planes are loaded only now: they do not occupy registers across the sub-step loop
  hot_epilogue_loaded<REF>(e, c, a, i, av);
}
template <bool REF>
QX_DI void hot_epilogue_loaded(Env& e, const DevConfig& c, const StepArgs& a, const int64_t i, const float4 av) {
  constexpr int OBS_DIM = QX_OBS_DIM_HOVER;
  const float act[4] = {av.x, av.y, av.z, av.w};
  float obs[OBS_DIM];
  ObsAux x;
  build_obs<QX_TASK_HOVER, false>(e, c, act, 0, true, obs, x);
  const bool done = reward_and_flags<QX_TASK_HOVER, false>(e, c, a, i, act, true, obs, x);
  if (done) episode_end<true>(e, a, i, obs);
  else if (a.obs) write_obs(obs, a.obs, i, a.obs_stride, a.obs_bf16 != 0, a.stream_stores != 0);
  if (a.stream_stores >= 2) store_env<true>(e, a.state, a.n, i);
  else store_env(e, a.state, a.n, i);
  if (done && a.merged) __threadfence();  // merged launch: the queue entry and these planes are read by a draining block
}

// reset of a queued env inside the merged launch: its planes were stored by this launch, so no read-only loads
template <bool REF>
__device__ __noinline__ void run_env_requeue(const DevConfig& cparam, const StepArgs& a, const int64_t i) {
  DevConfig cref = cparam;
  if (REF) apply_ref_constants(cref);
  const DevConfig& c = REF ? cref : cparam;
  run_env<MODE_RESET_QUEUE, QX_TASK_HOVER, false, false>(c, a, i);
}

// one agent step of envs i0 (and i1 when V has two lanes) in the calling thread
// V = float: one env per thread;  V = P2<true> / P2<false>: two envs per thread, packed / scalar arithmetic
// the 12 sub-steps of one agent step for the env(s) of the calling thread: setpoint scaling (hover.py:337-341), then per
// Aviary.step() the rate PID, one Philox call per env and two physics sub-steps.  V = float: one env per thread;
// V = P2<true> / P2<false>: two envs per thread, packed / scalar arithmetic.
template <class V>
QX_DI void hot_substeps(const DevConfig& c, Env& e0, Env& e1, const float4 av0, const float4 av1, const int64_t i0, const int64_t i1) {
  constexpr int kLanes = Lane<V>::N;
  typedef LaneOps<V> L;
  Core<V> p;
  L::pack(p, e0, e1);
  V sp[4];  // hover.py:337-341
  sp[0] = vmul(L::make(av0.x, av1.x), c.act_scale[0]);
  sp[1] = vmul(L::make(av0.y, av1.y), c.act_scale[1]);
  sp[2] = vmul(L::make(av0.z, av1.z), c.act_scale[2]);
  sp[3] = vfma(L::make(av0.w, av1.w), c.thrust_scale, c.thrust_bias);
  sp[3] = L::make(__saturatef(half_of<0>(sp[3])), __saturatef(half_of<1>(sp[3])));  // QuadX.update_control clips the mode-0 thrust command to [0, 1]
  const uint32_t k0a = c.seed_lo ^ (c.env_lo + (uint32_t)i0), k0b = c.seed_lo ^ (c.env_lo + (uint32_t)i1);
  const uint32_t k1a = c.seed_hi ^ (c.env_hi + (uint32_t)(((uint64_t)c.env_lo + (uint64_t)i0) >> 32));
  const uint32_t k1b = c.seed_hi ^ (c.env_hi + (uint32_t)(((uint64_t)c.env_lo + (uint64_t)i1) >> 32));
  const int nsub = c.n_sub_step;
#pragma unroll 1
  for (int j = 0; j < nsub; j += 2) {  // one Aviary.step(): rate PID, one Philox call per env, two physics sub-steps
    V apwm[4];
    control_update<V>(p, c, sp, apwm);
    V nz[4] = {splat<V>(0.f), splat<V>(0.f), splat<V>(0.f), splat<V>(0.f)};
    uint4 ba = make_uint4(0u, 0u, 0u, 0u), bb = ba;
    if (c.noise) {
      ba = env_philox(make_uint4((uint32_t)j >> 1, STREAM_STEP, e0.rng_ctr, 0u), k0a, k1a);
      if (kLanes == 2) bb = env_philox(make_uint4((uint32_t)j >> 1, STREAM_STEP, e1.rng_ctr, 0u), k0b, k1b);
      if constexpr (kLanes == 2) normal4_scaled<V>(make_uint2(ba.x, bb.x), make_uint2(ba.y, bb.y), c.noise_k, nz);
      else normal4_scaled<V>(ba.x, ba.y, c.noise_k, nz);
    }
    physics_substep<V>(p, c, apwm, nz, false);
    if (c.noise) {
      if constexpr (kLanes == 2) normal4_scaled<V>(make_uint2(ba.z, bb.z), make_uint2(ba.w, bb.w), c.noise_k, nz);
      else normal4_scaled<V>(ba.z, ba.w, c.noise_k, nz);
    }
    physics_substep<V>(p, c, apwm, nz, j + 2 == nsub);
  }
  unpack_lane<0>(e0, p);
  if (kLanes == 2) unpack_lane<1>(e1, p);
}

#ifndef QX_SWP
#define QX_SWP 0
#endif
#ifndef QX_DIAG
#define QX_DIAG 0
#endif
#ifndef QX_RESET_SWP
#define QX_RESET_SWP 0
#endif
// the paired sub-step loop: nsub sub-steps (even) towards a fixed setpoint, noise stream `stream`.  FLOOR = false is the
// speculative loop without the floor stand-in (physics_substep_s); returns the lowest pz it saw (+inf with FLOOR = true).
template <bool FLOOR = true, int SWP = QX_SWP>
QX_DI float substeps_s(const DevConfig& c, Env& e0, const f2 spxy, const float spz, const float thrust, const int nsub, const uint32_t stream, const int64_t i0) {
  CoreS p;
  pack_core_s(p, e0);
  float minz = __int_as_float(0x7f800000);
  const uint32_t k0 = c.seed_lo ^ (c.env_lo + (uint32_t)i0);
  const uint32_t k1 = c.seed_hi ^ (c.env_hi + (uint32_t)(((uint64_t)c.env_lo + (uint64_t)i0) >> 32));
  if constexpr (SWP == 0) {
#pragma unroll 1
  for (int j = 0; j < nsub; j += 2) {  // one Aviary.step(): rate PID, one Philox call, two physics sub-steps
    f2 apwm[2];
    control_update_s(p, c, spxy, spz, thrust, apwm);
    f2 nz[2] = {f2{0.f, 0.f}, f2{0.f, 0.f}};
    uint4 b = make_uint4(0u, 0u, 0u, 0u);
    if (c.noise) {
#if QX_DIAG == 2  // diagnostic build (timing only, wrong numbers): no Philox
      b = make_uint4(k0 + j, k1 ^ j, e0.rng_ctr * 0x9E3779B9u + j, k0 * 0x85EBCA6Bu + j);
#else
      b = env_philox(make_uint4((uint32_t)j >> 1, stream, e0.rng_ctr, 0u), k0, k1);
#endif
#if QX_DIAG == 1  // diagnostic build (timing only, wrong numbers): no Box-Muller
      nz[0] = vmul(f2{__uint_as_float(0x3f800000u | (b.x >> 9)) - 1.5f, __uint_as_float(0x3f800000u | (b.x << 14 >> 9)) - 1.5f}, 0.02f);
      nz[1] = vmul(f2{__uint_as_float(0x3f800000u | (b.y >> 9)) - 1.5f, __uint_as_float(0x3f800000u | (b.y << 14 >> 9)) - 1.5f}, 0.02f);
#else
      normal4_scaled_s(b.x, b.y, c.noise_k, nz);
#endif
    }
    physics_substep_s<FLOOR>(p, c, apwm, nz, false, minz);
#if QX_DIAG == 1
    if (c.noise) {
      nz[0] = vmul(f2{__uint_as_float(0x3f800000u | (b.z >> 9)) - 1.5f, __uint_as_float(0x3f800000u | (b.z << 14 >> 9)) - 1.5f}, 0.02f);
      nz[1] = vmul(f2{__uint_as_float(0x3f800000u | (b.w >> 9)) - 1.5f, __uint_as_float(0x3f800000u | (b.w << 14 >> 9)) - 1.5f}, 0.02f);
    }
#else
    if (c.noise) normal4_scaled_s(b.z, b.w, c.noise_k, nz);
#endif
    physics_substep_s<FLOOR>(p, c, apwm, nz, j + 2 == nsub, minz);
  }
  } else if constexpr (SWP == 1) {
  // software-pipelined noise: the Philox call of Aviary.step j + 1 is issued at the top of step j, where nothing depends on it,
  // so that its ~7 x 3 dependent integer operations fill the stalls of the control / physics chain instead of heading it
  uint4 b = make_uint4(0u, 0u, 0u, 0u);
  if (c.noise) b = env_philox(make_uint4(0u, stream, e0.rng_ctr, 0u), k0, k1);
#pragma unroll 1
  for (int j = 0; j < nsub; j += 2) {
    const uint4 bc = b;
    if (c.noise && j + 2 < nsub) b = env_philox(make_uint4(((uint32_t)j >> 1) + 1u, stream, e0.rng_ctr, 0u), k0, k1);
    f2 apwm[2];
    control_update_s(p, c, spxy, spz, thrust, apwm);
    f2 nz[2] = {f2{0.f, 0.f}, f2{0.f, 0.f}};
    if (c.noise) normal4_scaled_s(bc.x, bc.y, c.noise_k, nz);
    physics_substep_s<FLOOR>(p, c, apwm, nz, false, minz);
    if (c.noise) normal4_scaled_s(bc.z, bc.w, c.noise_k, nz);
    physics_substep_s<FLOOR>(p, c, apwm, nz, j + 2 == nsub, minz);
  }
  } else {
  // ... and the Box-Muller transform with it: the 8 scaled normals of step j + 1 are ready before step j ends
  f2 na[2] = {f2{0.f, 0.f}, f2{0.f, 0.f}}, nb[2] = {f2{0.f, 0.f}, f2{0.f, 0.f}};
  if (c.noise) {
    const uint4 b = env_philox(make_uint4(0u, stream, e0.rng_ctr, 0u), k0, k1);
    normal4_scaled_s(b.x, b.y, c.noise_k, na);
    normal4_scaled_s(b.z, b.w, c.noise_k, nb);
  }
#pragma unroll 1
  for (int j = 0; j < nsub; j += 2) {
    const f2 ca[2] = {na[0], na[1]}, cb[2] = {nb[0], nb[1]};
    if (c.noise && j + 2 < nsub) {
      const uint4 b = env_philox(make_uint4(((uint32_t)j >> 1) + 1u, stream, e0.rng_ctr, 0u), k0, k1);
      normal4_scaled_s(b.x, b.y, c.noise_k, na);
      normal4_scaled_s(b.z, b.w, c.noise_k, nb);
    }
    f2 apwm[2];
    control_update_s(p, c, spxy, spz, thrust, apwm);
    physics_substep_s<FLOOR>(p, c, apwm, ca, false, minz);
    physics_substep_s<FLOOR>(p, c, apwm, cb, j + 2 == nsub, minz);
  }
  }
  unpack_core_s(e0, p);
  return minz;
}
// hot_substeps for V = S1: one env per thread with its own components paired (qx_model.cuh, CoreS)
template <>
QX_DI void hot_substeps<S1>(const DevConfig& c, Env& e0, Env&, const float4 av0, const float4, const int64_t i0, const int64_t) {
  const f2 spxy = vmul(f2{av0.x, av0.y}, cpair(c.act_scale[0], c.act_scale[1]));  // hover.py:337-341
  const float spz = __fmul_rn(av0.z, c.act_scale[2]);
  const float thrust = __saturatef(fmaf(av0.w, c.thrust_scale, c.thrust_bias));  // QuadX.update_control clips the mode-0 thrust command to [0, 1]
  substeps_s(c, e0, spxy, spz, thrust, c.n_sub_step, STREAM_STEP, i0);
}
#ifndef QX_SPEC_FLOOR
#define QX_SPEC_FLOOR 1
#endif
#ifndef QX_PREFETCH_TAIL
#define QX_PREFETCH_TAIL 1
#endif
// The same with the floor stand-in speculated away (QX_SPEC_FLOOR): a warp none of whose envs rests on the floor or is predicted
// to come near it within this agent step runs the loop without the stand-in and checks afterwards that no pz went below
// floor_z; an env that fails the check (rare: the predictor is generous) reloads its loop planes -- nothing has been stored yet
// -- and runs the full loop.  Every other warp runs the full loop as before.  Bitwise equal to hot_substeps<S1> by construction;
// tests/test_gpu_properties.py holds it against the generic kernels.
QX_DI void hot_substeps_spec(const DevConfig& c, Env& e0, const StepArgs& a, const float4 av0, const int64_t i0) {
  const f2 spxy = vmul(f2{av0.x, av0.y}, cpair(c.act_scale[0], c.act_scale[1]));
  const float spz = __fmul_rn(av0.z, c.act_scale[2]);
  const float thrust = __saturatef(fmaf(av0.w, c.thrust_scale, c.thrust_bias));
  // predictor: where pz would be after this agent step at the current vertical speed, less 2 g T^2 / 2 (T = n_sub_step h)
  const float T = __fmul_rn((float)c.n_sub_step, c.h);
  const float reach = fmaf(fminf(e0.vz, 0.f), T, e0.pz) - __fmul_rn(__fmul_rn(c.g, T), T);
  const bool risky = e0.contact || !(reach > c.floor_z);
  const bool slow = __any_sync(__activemask(), risky);
  float minz = __int_as_float(0x7f800000);
  if (!slow) minz = substeps_s<false>(c, e0, spxy, spz, thrust, c.n_sub_step, STREAM_STEP, i0);
  const bool redo = minz < c.floor_z;
  if (slow || redo) {
    if (redo) load_env_loop(e0, a.state, a.n, i0);
    substeps_s<true>(c, e0, spxy, spz, thrust, c.n_sub_step, STREAM_STEP, i0);
  }
}

// reset() of one queued env on the paired code (hover.py:72-113: respawn, the idle Aviary.step()s with a zero setpoint, first
// observation): what run_env<MODE_RESET_QUEUE> does, in the register budget of the hot kernels.  NC = false inside the merged
// launch, whose own step phase stored the planes this reads.
template <bool NC>
QX_DI void hot_reset_env(const DevConfig& c, const StepArgs& a, const int64_t i) {
  constexpr int OBS_DIM = QX_OBS_DIM_HOVER;
  Env e;
  load_env<NC>(e, a.state, a.n, i);
  const uint32_t k0 = c.seed_lo ^ (c.env_lo + (uint32_t)i);
  const uint32_t k1 = c.seed_hi ^ (c.env_hi + (uint32_t)(((uint64_t)c.env_lo + (uint64_t)i) >> 32));
  respawn(e, c, k0, k1);
  // set_mode(0): zero setpoint.  The reset-queue launch is a latency chain of a few warps (~7 us for the 20 idle sub-steps, 0.3
  // instructions per clock); generating the noise of Aviary.step j + 1 during step j (QX_RESET_SWP = 2) measured no shorter
  substeps_s<true, QX_RESET_SWP>(c, e, f2{0.f, 0.f}, 0.f, 0.f, c.n_sub_reset, STREAM_RESET, i);
  const float act[4] = {0.f, 0.f, 0.f, 0.f};  // hover.py:101
  float obs[OBS_DIM];
  ObsAux x;
  build_obs<QX_TASK_HOVER, false>(e, c, act, 1, true, obs, x);
  if (a.obs) write_obs(obs, a.obs, i, a.obs_stride, a.obs_bf16 != 0);
  store_env(e, a.state, a.n, i);
}
template <bool REF>
__device__ __noinline__ void hot_reset_requeue(const DevConfig& cparam, const StepArgs& a, const int64_t i) {
  DevConfig cref = cparam;
  if (REF) apply_ref_constants(cref);
  const DevConfig& c = REF ? cref : cparam;
  hot_reset_env<false>(c, a, i);
}

// one agent step of envs i0 (and i1 when V has two lanes) in the calling thread, state and actions from global memory
template <bool REF, class V>
QX_DI void hot_task(const DevConfig& c, const DevConfig& cparam, const StepArgs& a, const int64_t i0, const int64_t i1, const bool has1) {
  constexpr int kLanes = Lane<V>::N;
  Env e0, e1;
  // the action is requested together with the state planes: loaded after the finished-env test below it cost every warp a second,
  // serialised trip to HBM (4.5 % of the warp's lifetime in the ncu stall samples of profiles/k1_r2k.md)
  const float4 av0 = __ldg(reinterpret_cast<const float4*>(a.actions) + i0);
  const float4 av1 = kLanes == 2 ? __ldg(reinterpret_cast<const float4*>(a.actions) + i1) : av0;
  load_env_loop(e0, a.state, a.n, i0);
  if (kLanes == 2) load_env_loop(e1, a.state, a.n, i1);
  if ((e0.flags | (kLanes == 2 ? e1.flags : 0u)) & (F_TERM | F_TRUNC)) {  // cold: a finished env does not step (hover.py:347-348)
    run_env_cold<REF>(cparam, a, i0);
    if (has1) run_env_cold<REF>(cparam, a, i1);
    return;
  }
#if QX_PREFETCH_TAIL
  // the epilogue planes are loaded after the loop (no registers across it); ask L2 for them now
#pragma unroll
  for (int p = kLoopPlanes; p < 11; ++p) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.state + (int64_t)p * a.n + i0));
#endif
  if constexpr (QX_SPEC_FLOOR && std::is_same<V, S1>::value) hot_substeps_spec(c, e0, a, av0, i0);
  else hot_substeps<V>(c, e0, e1, av0, av1, i0, i1);
  hot_epilogue<REF>(e0, c, a, i0, av0);
  if (has1) hot_epilogue<REF>(e1, c, a, i1, av1);
}

QX_DI unsigned int ld_acquire_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// The unit of work is a warp task: 32 x lanes consecutive envs (lane l of the warp owns env base + l, and base + 32 + l
// with two lanes); warp w of block b runs task b * warps + w.
//
// MERGED = false: the reset queue is drained by a second launch (MODE_RESET_QUEUE).
//
// MERGED = true (auto-reset): ONE launch per agent step.  Every block takes a ticket when it is done; the blocks holding
// the last `a.drainers` tickets (the last resident wave -- at most that many blocks can still be running or waiting
// when they arrive, so they all fit on the SMs and the wait below cannot deadlock) stay, wait until every block has
// retired, and drain the reset queue the step phase filled -- in full warps, like the separate launch, but without the
// second launch and the idle gap before it.  Only a thread that queued an env issues a fence (after its stores, before
// its block's ticket): the queue entry and that env's planes are all a drainer reads.  The last block to leave re-arms
// the counters for the next launch and publishes the queue length for qx_done_queue.
//
// Measured and rejected (B200, 1 Mi envs; profiles/k1_r2_merged.md): a persistent grid whose warps draw tasks from a
// counter -- 166 us against 139 + 8 us for two plain launches, long-scoreboard stalls doubled -- and the same with the
// next task's planes staged into shared memory by cp.async.bulk behind an mbarrier (174 us).
template <bool REF, int SHAPE, class V, bool MERGED>
__global__ void __launch_bounds__(HotShape<SHAPE>::kBlock, HotShape<SHAPE>::kMinBlocks) quadx_step_hot_kernel(const __grid_constant__ DevConfig cparam,
                                                                                                                 const __grid_constant__ StepArgs a) {
  constexpr int kB = HotShape<SHAPE>::kBlock, kLanes = Lane<V>::N, kWarps = kB / 32, kTask = 32 * kLanes;
  if constexpr (!MERGED) {
    // launched as a programmatic dependent of the kernel before it on the stream (launch_hot_kernel): wait for that grid and its
    // memory; then the reset-queue launch that follows may be scheduled as soon as the last wave of this grid has started
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
  }
  DevConfig cref = cparam;
  if (REF) apply_ref_constants(cref);
  const DevConfig& c = REF ? cref : cparam;
  const int64_t end = a.env_begin + a.env_count;
  const int64_t i0 = a.env_begin + ((int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5)) * kTask + (threadIdx.x & 31u);
  if (i0 < end) {
    const bool has1 = kLanes == 2 && i0 + 32 < end;
    hot_task<REF, V>(c, cparam, a, i0, has1 ? i0 + 32 : i0, has1);  // a thread without a second env computes its first one twice, stores it once
  }
  if constexpr (!MERGED) {
    if (a.queue) publish_queue_length(a.queue);  // two-launch step: the reset-queue launch follows
  }
  if constexpr (MERGED) {
    ResetQueue* const q = a.queue;
    __shared__ unsigned int s_ticket;
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(&q->tasks_done, 1u);
    __syncthreads();
    if (s_ticket + a.drainers < gridDim.x) return;
    if (threadIdx.x == 0) {
      unsigned int ns = 64u;
      while (ld_acquire_u32(&q->tasks_done) < gridDim.x) { __nanosleep(ns); if (ns < 512u) ns += ns; }
    }
    __syncthreads();
    const unsigned int cnt = ld_acquire_u32(&q->count);
#pragma unroll 1
    while (cnt != 0u) {
      unsigned int r = 0u;
      if ((threadIdx.x & 31u) == 0u) r = atomicAdd(&q->next_reset, 32u);
      r = __shfl_sync(0xffffffffu, r, 0);
      if (r >= cnt) break;
      if (r + (threadIdx.x & 31u) < cnt) {
        const int64_t ie = (int64_t)__ldcg(&q->idx[r + (threadIdx.x & 31u)]);
        if (a.paired_reset) hot_reset_requeue<REF>(cparam, a, ie);
        else run_env_requeue<REF>(cparam, a, ie);
      }
      __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      const unsigned int n_drain = a.drainers < gridDim.x ? a.drainers : gridDim.x;
      if (atomicAdd(&q->exit_ticket, 1u) == n_drain - 1u) {
        q->published = cnt; q->count = 0u; q->tasks_done = 0u; q->next_reset = 0u; q->exit_ticket = 0u;
      }
    }
  }
}

// MODE_RESET_QUEUE on the paired code: the second launch of the two-launch step
template <bool REF>
__global__ void __launch_bounds__(128, 4) quadx_reset_hot_kernel(const __grid_constant__ DevConfig cparam, const __grid_constant__ StepArgs a) {
  DevConfig cref = cparam;
  if (REF) apply_ref_constants(cref);
  const DevConfig& c = REF ? cref : cparam;
  // launched as a programmatic dependent of the step launch (qx_step): the blocks are already on the SMs when the step grid
  // retires and wait here for its memory; a no-op in a plain launch
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;");  // the next step launch of a tight loop (it waits at its own top)
  const unsigned int cnt = *reinterpret_cast<volatile unsigned int*>(&a.queue->count);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&a.queue->ticket, 1u) == gridDim.x - 1) { a.queue->count = 0u; a.queue->ticket = 0u; }
  }
  for (unsigned int t = blockIdx.x * 128 + threadIdx.x; t < cnt; t += gridDim.x * 128) hot_reset_env<true>(c, a, (int64_t)a.queue->idx[t]);
}

// debug / measurement hook: SM clock and wall clock of one thread, so that two samples give the average SM frequency
// of the interval between them (clock droop under sustained load does not show in NVML's slow readings)
__global__ void clock_probe_kernel(unsigned long long* out) {
  unsigned long long ns;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
  out[0] = (unsigned long long)clock64();
  out[1] = ns;
}

// ---------------------------------------------------------------------------
// K6: the FPV camera frame (qx_render).  One warp per 32-row band of a frame: lane l finds the covered columns of row
// band * 32 + l with the helpers vision_raster uses, so a frame holds exactly the pixels vision_mode = 1 counts; then the
// warp writes the band -- contiguous bytes of the frame -- with 16-byte stores, 512 contiguous bytes per store instruction.
// ---------------------------------------------------------------------------
constexpr int kRenderBlock = 256;
constexpr uint32_t kRgbaBox = 0xFF0000C8u, kRgbaSky = 0xFFE6BEAAu;  // (200, 0, 0, 255) and (170, 190, 230, 255), little-endian RGBA
struct RenderArgs {
  const float4* state;
  int64_t n;
  const int32_t* env_idx;  // nullable: frame f shows env f
  int64_t m;
  uint8_t* frames;
  int32_t res;
  const float* raster;     // RasterConsts
};

// The box crosses the near plane (vision_raster reports it unseen; a yawed drone can still have part of it in view): the
// silhouette is the projection of the box clipped to depth > cam_near, i.e. the convex hull of the corners in front and of the
// points where edges cross the plane.  Those points go to the warp's slice of shared memory (every lane computes the same);
// the hull's x interval on the row's centre line is the min / max over the vertex pairs crossing it (every such segment lies
// inside the hull and every hull edge is one of them).  Rare, so kept out of registers.
QX_DI void clipped_row_span(const RasterConsts& c, const float (&pxs)[8], const float (&pys)[8], const float (&xrs)[8], const float (&yus)[8],
                            const float (&deps)[8], float2* __restrict__ pts, const int row, int& ln, int& rn) {
  constexpr int ea[12] = {0, 1, 2, 3, 4, 5, 6, 7, 0, 1, 2, 3}, eb[12] = {1, 2, 3, 0, 5, 6, 7, 4, 4, 5, 6, 7};
  const int lane = threadIdx.x & 31;
  int nv = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (deps[k] > c.cam_near) {
      if (lane == 0) pts[nv] = make_float2(pxs[k], pys[k]);
      ++nv;
    }
  const float k1 = c.inv_tan / c.cam_near;
#pragma unroll
  for (int e = 0; e < 12; ++e) {
    const int a = ea[e], b = eb[e];
    if ((deps[a] > c.cam_near) != (deps[b] > c.cam_near)) {
      const float t = (c.cam_near - deps[a]) / (deps[b] - deps[a]);
      const float xr = fmaf(t, xrs[b] - xrs[a], xrs[a]), yu = fmaf(t, yus[b] - yus[a], yus[a]);
      if (lane == 0) pts[nv] = make_float2(fmaf(xr * k1, c.half_res, c.half_res), fmaf(-yu * k1, c.half_res, c.half_res));
      ++nv;
    }
  }
  __syncwarp();
  ln = 1; rn = 0;
  const float yl = (float)row + 0.5f;
  float xl = 3.0e38f, xr = -3.0e38f;
  for (int i = 1; i < nv; ++i) {
    const float2 p = pts[i];
    for (int j = 0; j < i; ++j) {
      const float2 q = pts[j];
      if ((p.y - yl) * (q.y - yl) <= 0.f && p.y != q.y) {
        const float xi = fmaf(yl - p.y, (q.x - p.x) / (q.y - p.y), p.x);
        xl = fminf(xl, xi); xr = fmaxf(xr, xi);
      }
    }
  }
  if (xl <= xr) { ln = (int)ceilf(xl - 0.5f); rn = (int)floorf(xr - 0.5f); }
}

// bits lo..hi (0 <= lo, hi <= 31) of a word; 0 when lo > hi
QX_DI uint32_t run_bits(int lo, int hi) { return lo > hi ? 0u : (0xFFFFFFFFu >> (31 - (hi - lo))) << lo; }

template <int FMT>
__global__ void __launch_bounds__(kRenderBlock) render_kernel(const __grid_constant__ RenderArgs a) {
  __shared__ float2 s_pts[kRenderBlock / 32][20];
  constexpr int C = FMT == QX_FRAME_RGBA ? 4 : 1, PPC = 16 / C;  // bytes per pixel, pixels per 16-byte chunk
  const int lane = threadIdx.x & 31, res = a.res, bands = (res + 31) >> 5;
  const int64_t warp = ((int64_t)blockIdx.x * kRenderBlock + threadIdx.x) >> 5;
  const int64_t f = warp / bands;
  if (f >= a.m) return;  // whole warps
  const int band = (int)(warp - f * bands);
  const int64_t i = a.env_idx ? (int64_t)a.env_idx[f] : f;
  int ln = 1, rn = 0;  // covered columns of row band * 32 + lane
  if (i >= 0 && i < a.n) {
    const RasterConsts c = *reinterpret_cast<const RasterConsts*>(a.raster);
    const float4 p0 = a.state[i], p1 = a.state[a.n + i];  // (px py pz qx) (qy qz qw ..)
    float pxs[8], pys[8], xrs[8], yus[8], deps[8];
    if (raster_project(c, p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, pxs, pys, xrs, yus, deps)) {
      RasterEdges E;
      raster_edges(pxs, pys, E);
      raster_row_span(E, band * 32 + lane, ln, rn);
    } else {
      clipped_row_span(c, pxs, pys, xrs, yus, deps, s_pts[threadIdx.x >> 5], band * 32 + lane, ln, rn);
    }
    ln = max(ln, 0); rn = min(rn, res - 1);  // (the float -> int conversions saturate far outside the image)
  }
  const int rows = min(32, res - band * 32);
  const int chunks = rows * res * C / 16;  // whole: res % 4 == 0
  uint4* out = reinterpret_cast<uint4*>(a.frames + ((f * res + band * 32) * res) * C);
  for (int c0 = 0; c0 < chunks; c0 += 32) {
    const int ch = c0 + lane, p = ch * PPC, r = p / res, col = p - r * res;  // first pixel of the chunk: row r (of the band), column col
    // a mask chunk runs into the next row when res % 16 != 0
    const int l0 = __shfl_sync(0xFFFFFFFFu, ln, r & 31), r0 = __shfl_sync(0xFFFFFFFFu, rn, r & 31);
    const int l1 = __shfl_sync(0xFFFFFFFFu, ln, (r + 1) & 31), r1 = __shfl_sync(0xFFFFFFFFu, rn, (r + 1) & 31);
    if (ch >= chunks) continue;
    const int wrap = res - col;  // pixels of the chunk still in row r
    uint32_t bits = run_bits(max(l0 - col, 0), min(min(r0 - col, wrap - 1), PPC - 1));
    if (wrap < PPC) bits |= run_bits(max(l1 + wrap, wrap), min(r1 + wrap, PPC - 1));
    uint4 v;
    if (FMT == QX_FRAME_RGBA) {
      v.x = bits & 1u ? kRgbaBox : kRgbaSky; v.y = bits & 2u ? kRgbaBox : kRgbaSky;
      v.z = bits & 4u ? kRgbaBox : kRgbaSky; v.w = bits & 8u ? kRgbaBox : kRgbaSky;
    } else {  // 4 bits -> 4 bytes of 0 / 255
      v.x = ((bits & 0xFu) * 0x00204081u & 0x01010101u) * 255u;
      v.y = ((bits >> 4 & 0xFu) * 0x00204081u & 0x01010101u) * 255u;
      v.z = ((bits >> 8 & 0xFu) * 0x00204081u & 0x01010101u) * 255u;
      v.w = ((bits >> 12 & 0xFu) * 0x00204081u & 0x01010101u) * 255u;
    }
    __stcs(out + ch, v);
  }
}

// ---------------------------------------------------------------------------
// K7: the evaluation ledger (qx_episode_record).  One thread per env, after every step of a handle without auto-reset: an
// open record whose env's flags word says the episode ended is closed with the return and length the state holds at that
// step -- later steps of the frozen env keep adding to ep_ret and step_count, so the result exists only on this step.  An
// open record costs one 16-byte load (plane 7), a closing one a second (plane 8), a closed one only its own end word.
// ---------------------------------------------------------------------------
constexpr int kRecordBlock = 256;
__global__ void __launch_bounds__(kRecordBlock) episode_record_kernel(const float4* __restrict__ state, const int64_t n, float* __restrict__ ret,
                                                                      int32_t* __restrict__ len, uint32_t* __restrict__ end,
                                                                      uint32_t* __restrict__ n_closed) {
  const int64_t i = (int64_t)blockIdx.x * kRecordBlock + threadIdx.x;
  if (i >= n || end[i] != 0u) return;
  const float4 p7 = state[7 * n + i];  // (svb2, step_count, rng_ctr, flags)
  const uint32_t fl = __float_as_uint(p7.w);
  if (!(fl & (F_TERM | F_TRUNC))) return;
  ret[i] = state[8 * n + i].w;  // (peul0, peul1, peul2, ep_ret)
  len[i] = __float_as_int(p7.y);
  end[i] = fl;
  // envs that end together (a mass floor termination) count with one atomic per warp, as episode_end does
  const auto g = cooperative_groups::coalesced_threads();
  if (g.thread_rank() == 0) atomicAdd(n_closed, g.size());
}

}  // namespace qx

// ===========================================================================
// host side / C-ABI
// ===========================================================================
struct QxHandle {
  QxConfig cfg;
  qx::DevConfig dev;
  int64_t n;
  int device;
  int planes;  // float4 state planes: 11, or 17 when flight_mode != 0
  bool ref_constants;  // the model constants equal the reference's literals bit for bit: run the specialised kernels
  bool hot_ok;         // hover, flight mode 0, control every 2nd sub-step: the lean one-step kernel applies
  int hot_mode;        // QX_HOT env var at qx_create: -1 default (large batches), 0 never, 1 always
  int paired_reset;    // QX_PAIRED_RESET (default 1 where it applies): queued envs are re-created by the paired code in the hot kernels' register budget
  int hot_lanes;       // QX_LANES: 1 one env per thread (scalar), 2 two envs per thread on packed f32x2, 4 one env per thread with its own components paired (f32x2)
  int hot_shape;       // QX_SHAPE: launch shape (HotShape)
  int stream_stores;   // QX_STREAM_STORES: 0 plain stores, 1 evict-first for obs / reward / flags, 2 also for the state planes
  int merged;          // QX_MERGED: 1 (default) the hot kernel also drains the reset queue (one launch per step), 0 separate reset launch
  int sm_count;
  int pdl;             // QX_PDL (default 1): qx_step launches the reset-queue kernel as a programmatic dependent of the step kernel
  int host_chunks;     // QX_HOST_CHUNKS: 0 (default) = the geometric piece schedule of the *_host calls, k > 0 = k equal pieces, the first halved again
  int host_one_d2h;    // QX_HOST_ONE_D2H: the small result arrays share the observation's D2H stream
  int hot_grid;        // blocks of one resident wave of the merged launch (SMs x blocks per SM from the occupancy calculator), 0 = not computed yet
  float4* state;
  qx::Stats* stats;
  qx::ResetQueue* queue;
  float* raster;       // vision_mode 1: qx::RasterConsts
  // staging for the *_host calls
  cudaStream_t stream, h2d_stream, d2h_stream, d2h2_stream;  // d2h2: the small result arrays, so that their per-copy latency hides behind the observation copy
  cudaEvent_t ev_h2d[16], ev_k[16], ev_d2h;
  float* h_act; float* d_act;
  float* h_obs; float* d_obs;
  float* h_rew; float* d_rew;
  uint8_t* h_flags; uint8_t* d_flags;  // [2n] terminated | truncated, then [n] mask
  float* h_tobs; float* d_tobs;
  bool staging;
};

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

// shared with ppo_kernels.cu (qx_internal.h): record the calling thread's last error, return the code
int qx_fail(int code, const char* fmt, const char* detail) {
  snprintf(g_err, sizeof(g_err), fmt, detail);
  return code;
}
static int fail(int code, const char* fmt, const char* detail = "") { return qx_fail(code, fmt, detail); }
#define QX_CUDA(call)                                                             \
  do {                                                                            \
    cudaError_t _e = (call);                                                      \
    if (_e != cudaSuccess) return fail(QX_ECUDA, #call ": %s", cudaGetErrorString(_e)); \
  } while (0)

extern "C" const char* qx_last_error(void) { return g_err; }
extern "C" int32_t qx_version(void) { return QX_VERSION; }
extern "C" int64_t qx_launch_count(void) { return g_launches.load(); }
extern "C" int64_t qx_sizeof_config(void) { return (int64_t)sizeof(QxConfig); }

extern "C" int qx_default_config(int32_t task, QxConfig* c) {
  if (!c || (task != QX_TASK_HOVER && task != QX_TASK_YAW)) return fail(QX_EINVAL, "qx_default_config: bad arguments");
  memset(c, 0, sizeof(*c));
  c->task = task;
  c->mass = 0.1f;
  c->inertia[0] = 3e-5f; c->inertia[1] = 3e-5f; c->inertia[2] = 5e-5f;
  const float mx[4] = {0.028f, -0.028f, 0.028f, -0.028f}, my[4] = {-0.028f, 0.028f, 0.028f, -0.028f};
  const float ts[4] = {-1.f, -1.f, 1.f, 1.f};
  const float map[16] = {-1, -1, -1, 1, 1, 1, -1, 1, 1, -1, 1, 1, -1, 1, 1, 1};
  memcpy(c->motor_x, mx, sizeof(mx)); memcpy(c->motor_y, my, sizeof(my));
  memcpy(c->torque_sign, ts, sizeof(ts)); memcpy(c->motor_map, map, sizeof(map));
  c->total_thrust = 4.0f; c->thrust_coef = 3.16e-10f; c->torque_coef = 7.94e-12f; c->noise_ratio = 0.02f; c->tau = 0.01f;
  c->drag_coef_xyz = 1.5f; c->drag_area_xyz = 3.0e-4f; c->drag_coef_pqr = 1.0e-4f; c->air_density = 1.225f;
  const float kp[3] = {2.0e-2f, 2.0e-2f, 4.0e-2f}, ki[3] = {2.5e-7f, 2.5e-7f, 1.35e-4f}, kd[3] = {5.0e-5f, 5.0e-5f, 0.f};
  for (int a = 0; a < 3; ++a) { c->rate_kp[a] = kp[a]; c->rate_ki[a] = ki[a]; c->rate_kd[a] = kd[a]; c->rate_lim[a] = 1.0f; }
  c->pwm_idle = 0.05f; c->physics_hz = 240.f; c->control_hz = 120.f; c->gravity = 9.81f;
  c->state_stale = 1; c->gyro = 1; c->max_coord_vel = 100.f; c->floor_z = 0.01f;
  c->cam_tilt_up_deg = 25.f; c->cam_fov_deg = 90.f; c->cam_res = 128.f; c->cam_near = 0.1f; c->vis_margin_px = 0.5f;
  const float panel[12] = {4.98f, -1, 5, 4.98f, 1, 5, 4.98f, 1, 7, 4.98f, -1, 7};
  memcpy(c->panel, panel, sizeof(panel));
  for (int k = 0; k < 4; ++k) { c->panel_back[3 * k] = panel[3 * k] + 0.04f; c->panel_back[3 * k + 1] = panel[3 * k + 1]; c->panel_back[3 * k + 2] = panel[3 * k + 2]; }  /* hover.py:118-147: box half extent 0.02 in depth */
  c->vision_mode = 0;
  c->aviary_steps_per_step = task == QX_TASK_HOVER ? 6 : 1;
  c->max_steps = 400; c->floor_grace_steps = 30; c->reset_idle_steps = task == QX_TASK_HOVER ? 10 : 0;
  c->agent_dt = 0.025f; c->flight_dome_size = 3.0f; c->floor_threshold = 0.1f;
  c->target_area = 0.013f; c->target_ratio = 1.53f;
  c->action_scale[0] = 30.f; c->action_scale[1] = 30.f; c->action_scale[2] = -30.f;
  c->spawn_yaw_noise = task == QX_TASK_YAW ? 3.14159265f : 0.f;  /* yaw.py:79 U(-pi, pi) */
  if (task == QX_TASK_YAW) {
    /* main.py:8-23 / yaw.py: default PyFlyt camera (camera_angle_degrees = +20), red sphere at (2, 0, 1), one Aviary.step per
       env step.  Sign: hover.py's camera_angle_degrees = -25 is read as 25 deg UP (DESIGN 4: the only reading under which the
       panel and the reference's target_area / target_ratio are in view), i.e. PyFlyt's positive angle points DOWN -- so the
       default +20 is 20 deg down.  From the ground (yaw.py never lifts off) the sphere then sits just above the image. */
    c->cam_tilt_up_deg = -20.f;
    c->panel[0] = 2.f; c->panel[1] = 0.f; c->panel[2] = 1.f;
    c->agent_dt = 1.0f / 120.f;
  }
  c->render = 0; c->auto_reset = 1; c->noise = 1;
  c->flight_mode = 0; c->thrust_scale = 0.5f; c->thrust_bias = 0.5f;  /* hover.py:92, :341 */
  const float att[12] = {1, 1, 1, 0, 0, 0, 0, 0, 0, 2, 2, 2};                                  /* cf2x.yaml:21-26 */
  const float vel[8] = {0.4f, 0.4f, 0.15f, 0.15f, 0.25f, 0.25f, 0.3f, 0.3f};                   /* cf2x.yaml:28-33 */
  const float pos[8] = {0.5f, 0.5f, 0, 0, 0, 0, 1, 1};                                         /* cf2x.yaml:35-40 */
  const float zp[4] = {0.8f, 0, 0, 1.5f}, zv[4] = {1.5f, 0.3f, 0.05f, 1.0f};                   /* cf2x.yaml:42-54 */
  memcpy(c->att_pid, att, sizeof(att)); memcpy(c->vel_pid, vel, sizeof(vel)); memcpy(c->pos_pid, pos, sizeof(pos));
  memcpy(c->zpos_pid, zp, sizeof(zp)); memcpy(c->zvel_pid, zv, sizeof(zv));
  return QX_OK;
}

static int derive(const QxConfig& s, uint64_t seed, uint64_t env_id0, qx::DevConfig* d) {
  memset(d, 0, sizeof(*d));
  if (s.task != QX_TASK_HOVER && s.task != QX_TASK_YAW) return fail(QX_EINVAL, "qx_create: unknown task");
  if (!(s.physics_hz > 0) || !(s.control_hz > 0) || s.control_hz > s.physics_hz) return fail(QX_EINVAL, "qx_create: bad rates");
  if (s.flight_mode < -1 || s.flight_mode > 7) return fail(QX_EINVAL, "qx_create: flight_mode outside PyFlyt's -1..7");
  if (s.flight_mode != 0 && s.task != QX_TASK_HOVER) return fail(QX_EINVAL, "qx_create: flight modes other than 0 apply to the hover task");
  if (s.vision_mode != 0 && s.vision_mode != 1) return fail(QX_EINVAL, "qx_create: vision_mode is 0 (analytic) or 1 (raster)");
  const int per = (int)(s.physics_hz / s.control_hz);
  d->task = s.task;
  d->ctrl_every = per;
  d->n_sub_step = s.aviary_steps_per_step * per;
  d->n_sub_reset = s.reset_idle_steps * per;
  d->max_steps = s.max_steps; d->floor_grace = s.floor_grace_steps; d->render = s.render; d->auto_reset = s.auto_reset;
  d->noise = (s.noise && s.noise_ratio != 0.f) ? 1 : 0;
  d->state_stale = s.state_stale; d->gyro = s.gyro;
  d->obs_dim = s.task == QX_TASK_HOVER ? QX_OBS_DIM_HOVER : QX_OBS_DIM_YAW;
  d->act_dim = s.task == QX_TASK_HOVER ? QX_ACT_DIM_HOVER : QX_ACT_DIM_YAW;
  const double h = 1.0 / s.physics_hz, T = 1.0 / s.control_hz;
  d->h = (float)h; d->lag_alpha = (float)(h / s.tau); d->one_m_alpha = (float)(1.0 - h / s.tau); d->noise_ratio = s.noise_ratio;
  d->noise_k = (float)(-2.0 * M_LN2 * (double)s.noise_ratio * (double)s.noise_ratio);
  d->thrust_k = (float)(s.total_thrust / 4.0); d->pwm_idle = s.pwm_idle;
  const double max_rpm2 = s.total_thrust / (4.0 * s.thrust_coef);
  for (int m = 0; m < 4; ++m) {
    d->torque_k[m] = (float)(s.torque_sign[m] * s.torque_coef * max_rpm2);
    d->mx[m] = s.motor_x[m]; d->my[m] = s.motor_y[m];
  }
  memcpy(d->map, s.motor_map, sizeof(d->map));
  d->drag_c = (float)(0.5 * s.air_density * s.drag_coef_xyz * s.drag_area_xyz); d->drag_pqr = s.drag_coef_pqr;
  for (int a = 0; a < 3; ++a) {
    d->kp[a] = s.rate_kp[a]; d->kiT[a] = (float)(s.rate_ki[a] * T); d->kd_T[a] = (float)(s.rate_kd[a] / T); d->lim[a] = s.rate_lim[a];
    d->I[a] = s.inertia[a]; d->invI[a] = (float)(1.0 / s.inertia[a]);
    d->cam_off[a] = s.cam_offset[a]; d->act_scale[a] = s.action_scale[a];
    d->start_pos[a] = s.start_pos[a]; d->start_rpy[a] = s.start_rpy[a];
  }
  d->inv_mass = (float)(1.0 / s.mass); d->g = s.gravity; d->vmax = s.max_coord_vel; d->floor_z = s.floor_z;
  for (int a = 0; a < 3; ++a) {
    d->hI[a] = (float)(h / s.inertia[a]);
    d->gk[a] = s.gyro ? (float)(-(h / s.inertia[a]) * ((double)s.inertia[(a + 2) % 3] - (double)s.inertia[(a + 1) % 3])) : 0.f;
  }
  d->hm = (float)(h / s.mass); d->hg = (float)(h * s.gravity); d->hh = (float)(0.5 * h); d->hh2 = (float)(0.25 * h * h);
  d->kq1 = (float)(-0.5 * h / 6.0); d->kq2 = (float)(0.5 * h / 120.0);
  d->ndrag_c = -(float)(0.5 * s.air_density * s.drag_coef_xyz * s.drag_area_xyz); d->ndrag_pqr = -s.drag_coef_pqr;
  const double tilt = s.cam_tilt_up_deg * M_PI / 180.0;
  d->cam_sd = (float)sin(tilt); d->cam_cd = (float)cos(tilt);
  d->inv_tan = (float)(1.0 / tan(0.5 * s.cam_fov_deg * M_PI / 180.0));
  d->res = s.cam_res; d->half_res = 0.5f * s.cam_res; d->inv_half_res = 2.0f / s.cam_res; d->inv_res2 = 1.0f / (s.cam_res * s.cam_res);
  d->cam_near = s.cam_near; d->margin = s.vis_margin_px;
  memcpy(d->panel, s.panel, sizeof(d->panel));
  d->vision_mode = s.vision_mode;
  d->inv_agent_dt = 1.0f / s.agent_dt; d->dome2 = s.flight_dome_size * s.flight_dome_size; d->floor_thr = s.floor_threshold;
  d->target_area = s.target_area; d->target_ratio = s.target_ratio;
  d->spawn_thr = s.spawn_throttle; d->spawn_pos_noise = s.spawn_pos_noise; d->spawn_yaw_noise = s.spawn_yaw_noise;
  d->seed_lo = (uint32_t)seed; d->seed_hi = (uint32_t)(seed >> 32);
  d->env_lo = (uint32_t)env_id0; d->env_hi = (uint32_t)(env_id0 >> 32);
  d->flight_mode = s.flight_mode; d->need_euler = (s.flight_mode == 1 || s.flight_mode == 3 || s.flight_mode >= 4) ? 1 : 0;
  d->thrust_scale = s.thrust_scale; d->thrust_bias = s.thrust_bias;
  auto gains = [T](const float* src, int w, float* dst) {  // kp | ki T | kd / T | lim
    for (int k = 0; k < w; ++k) {
      dst[k] = src[k]; dst[w + k] = (float)(src[w + k] * T); dst[2 * w + k] = (float)(src[2 * w + k] / T); dst[3 * w + k] = src[3 * w + k];
    }
  };
  gains(s.att_pid, 3, d->att); gains(s.vel_pid, 2, d->vel); gains(s.pos_pid, 2, d->lpos); gains(s.zpos_pid, 1, d->zpos); gains(s.zvel_pid, 1, d->zvel);
  // motor geometry folded with the thrust scale; symmetric-X shortcuts when the config allows them (cf2x.urdf:35-68 does)
  for (int m = 0; m < 4; ++m) { d->arm_x[m] = -d->thrust_k * d->mx[m]; d->arm_y[m] = d->thrust_k * d->my[m]; }
  const float ax = d->mx[0], tq = d->torque_k[2];
  d->x_layout = (ax > 0.f && d->mx[1] == -ax && d->mx[2] == ax && d->mx[3] == -ax && d->my[0] == -ax && d->my[1] == ax && d->my[2] == ax &&
                 d->my[3] == -ax && d->torque_k[0] == -tq && d->torque_k[1] == -tq && d->torque_k[3] == tq) ? 1 : 0;
  d->arm_k = d->thrust_k * ax; d->tq_k = tq;
  static const float xmap[16] = {-1, -1, -1, 1, 1, 1, -1, 1, 1, -1, 1, 1, -1, 1, 1, 1};
  d->x_mixer = memcmp(d->map, xmap, sizeof(xmap)) == 0 ? 1 : 0;
  return QX_OK;
}

static bool matches_ref_constants(const qx::DevConfig& d);
constexpr int kDefaultHotLanes = 4, kDefaultShape1 = 4, kDefaultShape2 = 0;  // measured on B200, profiles/k1_r2_variants.md

extern "C" int qx_create(const QxConfig* cfg, int64_t n_envs, uint64_t seed, uint64_t env_id0, int device, QxHandle** out) {
  if (!cfg || !out || n_envs <= 0) return fail(QX_EINVAL, "qx_create: bad arguments");
  int ndev = 0;
  QX_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(QX_EINVAL, "qx_create: no such device");
  cudaDeviceProp prop;
  QX_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(QX_EARCH, "qx_create: this library is built for sm_100a (B200) only");
  QxHandle* h = new (std::nothrow) QxHandle();
  if (!h) return fail(QX_ENOMEM, "qx_create: out of host memory");
  memset(h, 0, sizeof(*h));
  h->cfg = *cfg; h->n = n_envs; h->device = device;
  int rc = derive(*cfg, seed, env_id0, &h->dev);
  if (rc) { delete h; return rc; }
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(device);
  h->planes = cfg->flight_mode != 0 ? qx::kCascadePlanes : qx::kBasePlanes;
  h->ref_constants = !getenv("QX_FORCE_GENERIC") && matches_ref_constants(h->dev);
  h->hot_ok = cfg->task == QX_TASK_HOVER && cfg->flight_mode == 0 && cfg->vision_mode == 0 && h->dev.ctrl_every == 2 && (h->dev.n_sub_step & 1) == 0 && h->dev.n_sub_step > 0;
  auto env_int = [](const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; };
  h->hot_mode = env_int("QX_HOT", -1);
  h->hot_lanes = env_int("QX_LANES", kDefaultHotLanes);
  if (h->hot_lanes != 1 && h->hot_lanes != 2 && h->hot_lanes != 4) h->hot_lanes = kDefaultHotLanes;
  if (h->hot_lanes == 4 && !(cfg->spawn_throttle >= 0.f && cfg->pwm_idle >= 0.f)) h->hot_lanes = 1;  // the paired code assumes throttles >= 0
  h->hot_shape = env_int("QX_SHAPE", h->hot_lanes != 2 ? kDefaultShape1 : kDefaultShape2);
  if (h->hot_shape < 0 || h->hot_shape >= qx::kHotShapes || h->hot_shape == 1 || h->hot_shape == 2) h->hot_shape = h->hot_lanes != 2 ? kDefaultShape1 : kDefaultShape2;
  h->paired_reset = (h->hot_ok && (h->dev.n_sub_reset & 1) == 0 && cfg->spawn_throttle >= 0.f && cfg->pwm_idle >= 0.f && env_int("QX_PAIRED_RESET", 1)) ? 1 : 0;
  h->pdl = env_int("QX_PDL", 1);
  h->host_chunks = env_int("QX_HOST_CHUNKS", 0);
  if (h->host_chunks < -8 || h->host_chunks > 15 || h->host_chunks == -1) h->host_chunks = 0;
  h->host_one_d2h = env_int("QX_HOST_ONE_D2H", 0);
  h->merged = env_int("QX_MERGED", 0);  // measured: saves the second launch (~5 us) when nothing finishes, loses ~13 us when the queue is not empty
  h->sm_count = prop.multiProcessorCount;
  h->stream_stores = env_int("QX_STREAM_STORES", 0);
  cudaError_t e = cudaMalloc(&h->state, sizeof(float4) * h->planes * n_envs);
  if (e == cudaSuccess) e = cudaMalloc(&h->stats, sizeof(qx::Stats));
  if (e == cudaSuccess) e = cudaMalloc(&h->queue, sizeof(qx::ResetQueue) + sizeof(unsigned int) * n_envs);
  if (e == cudaSuccess) e = cudaMemset(h->queue, 0, sizeof(qx::ResetQueue));
  if (e == cudaSuccess) e = cudaMemset(h->state, 0, sizeof(float4) * h->planes * n_envs);
  if (e == cudaSuccess) e = cudaMemset(h->stats, 0, sizeof(qx::Stats));
  if (e == cudaSuccess) e = cudaMalloc(&h->raster, sizeof(qx::RasterConsts));
  if (e == cudaSuccess) {
    const qx::DevConfig& d = h->dev;
    qx::RasterConsts rc = {d.cam_sd, d.cam_cd, d.inv_tan, d.res, d.half_res, d.inv_half_res, d.inv_res2, d.cam_near, {d.cam_off[0], d.cam_off[1], d.cam_off[2]}, 0.f, {}, {}};
    memcpy(rc.panel, cfg->panel, sizeof(rc.panel)); memcpy(rc.panel_back, cfg->panel_back, sizeof(rc.panel_back));
    e = cudaMemcpy(h->raster, &rc, sizeof(rc), cudaMemcpyHostToDevice);
    h->dev.raster = h->raster;
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->d2h2_stream, cudaStreamNonBlocking);
  for (int k = 0; k < 16 && e == cudaSuccess; ++k) {
    e = cudaEventCreateWithFlags(&h->ev_h2d[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_k[k], cudaEventDisableTiming);
  }
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_d2h, cudaEventDisableTiming);
  cudaSetDevice(prev);
  if (e != cudaSuccess) {
    cudaFree(h->state); cudaFree(h->stats); cudaFree(h->queue); cudaFree(h->raster); delete h;
    return fail(QX_ECUDA, "qx_create: %s", cudaGetErrorString(e));
  }
  *out = h;
  return QX_OK;
}

extern "C" int qx_destroy(QxHandle* h) {
  if (!h) return QX_OK;
  int prev = 0;
  cudaGetDevice(&prev);
  cudaSetDevice(h->device);
  cudaFree(h->state); cudaFree(h->stats); cudaFree(h->queue); cudaFree(h->raster);
  if (h->staging) {
    cudaFreeHost(h->h_act); cudaFreeHost(h->h_obs); cudaFreeHost(h->h_rew); cudaFreeHost(h->h_flags); cudaFreeHost(h->h_tobs);
    cudaFree(h->d_act); cudaFree(h->d_obs); cudaFree(h->d_rew); cudaFree(h->d_flags); cudaFree(h->d_tobs);
  }
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->h2d_stream) cudaStreamDestroy(h->h2d_stream);
  if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
  if (h->d2h2_stream) cudaStreamDestroy(h->d2h2_stream);
  for (int k = 0; k < 16; ++k) { if (h->ev_h2d[k]) cudaEventDestroy(h->ev_h2d[k]); if (h->ev_k[k]) cudaEventDestroy(h->ev_k[k]); }
  if (h->ev_d2h) cudaEventDestroy(h->ev_d2h);
  cudaSetDevice(prev);
  delete h;
  return QX_OK;
}

struct DeviceGuard {
  int prev = 0;
  explicit DeviceGuard(int d) { cudaGetDevice(&prev); cudaSetDevice(d); }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

extern "C" int qx_nonfinite_count(QxHandle* h, int64_t* count) {
  if (!h || !count) return fail(QX_EINVAL, "qx_nonfinite_count: bad arguments");
  DeviceGuard g(h->device);
  qx::Stats s;
  QX_CUDA(cudaMemcpy(&s, h->stats, sizeof(s), cudaMemcpyDeviceToHost));
  *count = (int64_t)s.n_nonfinite;
  return QX_OK;
}

extern "C" int64_t qx_num_envs(const QxHandle* h) { return h ? h->n : 0; }
extern "C" int32_t qx_obs_dim(const QxHandle* h) { return h ? h->dev.obs_dim : 0; }
extern "C" int32_t qx_act_dim(const QxHandle* h) { return h ? h->dev.act_dim : 0; }
extern "C" void* qx_state_ptr(QxHandle* h) { return h ? h->state : nullptr; }
extern "C" int32_t qx_state_words(const QxHandle* h) { return h ? 4 * h->planes : 0; }
static bool matches_ref_constants(const qx::DevConfig& d) {
  qx::DevConfig lit = d;
  qx::apply_ref_constants(lit);
  return QX_HAVE_REF_CONSTANTS && d.task == QX_TASK_HOVER && d.flight_mode == 0 && memcmp(&lit, &d, sizeof(lit)) == 0;
}
extern "C" int32_t qx_uses_reference_constants(const QxHandle* h) { return h && h->ref_constants ? 1 : 0; }
// does this config take the specialised kernels?  (no GPU needed; -1 on a bad config)
extern "C" int32_t qx_config_matches_reference_constants(const QxConfig* cfg) {
  qx::DevConfig d;
  if (!cfg || derive(*cfg, 0, 0, &d) != QX_OK) return -1;
  return matches_ref_constants(d) ? 1 : 0;
}
// generator / test hook (not in the public header): the kernel-side constants derive() makes of a config; needs no GPU
extern "C" int64_t qx_debug_dev_config(const QxConfig* cfg, uint64_t seed, uint64_t env_id0, void* out, int64_t cap) {
  qx::DevConfig d;
  if (!cfg || derive(*cfg, seed, env_id0, &d) != QX_OK) return -1;
  if (out && cap >= (int64_t)sizeof(d)) memcpy(out, &d, sizeof(d));
  return (int64_t)sizeof(d);
}

template <int TASK, bool CASC, bool REF>
static void launch_task(QxHandle* h, int mode, const qx::StepArgs& a, cudaStream_t s) {
  const unsigned grid = (unsigned)((a.env_count + qx::kBlock - 1) / qx::kBlock);
  switch (mode) {
    case qx::MODE_STEP_INLINE:
      if (h->pdl) {  // one launch per agent step: consecutive steps chain as programmatic dependents (the kernel waits for its predecessor at its top)
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3(grid); lc.blockDim = dim3(qx::kBlock); lc.dynamicSmemBytes = 0; lc.stream = s;
        cudaLaunchAttribute at{};
        at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at.val.programmaticStreamSerializationAllowed = 1;
        lc.attrs = &at; lc.numAttrs = 1;
        cudaLaunchKernelEx(&lc, qx::quadx_step_kernel<qx::MODE_STEP_INLINE, TASK, CASC, REF>, h->dev, a);
      } else {
        qx::quadx_step_kernel<qx::MODE_STEP_INLINE, TASK, CASC, REF><<<grid, qx::kBlock, 0, s>>>(h->dev, a);
      }
      break;
    case qx::MODE_STEP_DEFER: qx::quadx_step_kernel<qx::MODE_STEP_DEFER, TASK, CASC, REF><<<grid, qx::kBlock, 0, s>>>(h->dev, a); break;
    case qx::MODE_RESET_MASK: qx::quadx_step_kernel<qx::MODE_RESET_MASK, TASK, CASC, REF><<<grid, qx::kBlock, 0, s>>>(h->dev, a); break;
    default: {
      const unsigned g = grid < (unsigned)qx::kResetQueueBlocks ? grid : (unsigned)qx::kResetQueueBlocks;
      qx::quadx_step_kernel<qx::MODE_RESET_QUEUE, TASK, CASC, REF><<<g, qx::kBlock, 0, s>>>(h->dev, a);
      break;
    }
  }
}

// The large-batch kernels join the programmatic launch chain only outside stream capture: inside the two-branch rollout graph
// (ppo.RolloutEngine) programmatic edges on the env-step and reset-queue nodes measured 1 % slower (3.04 vs 3.01 ms per
// 131 072 x 32 rollout), in a plain stream they save 3.6-4.3 us per step.  Single-launch steps chain in both (tools/small_ab.py).
static bool stream_is_capturing(cudaStream_t s) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  return cudaStreamIsCapturing(s, &st) == cudaSuccess && st != cudaStreamCaptureStatusNone;
}

template <bool REF, int SHAPE, class V>
static cudaError_t launch_hot_kernel(QxHandle* h, const qx::StepArgs& a, cudaStream_t s) {
  constexpr int B = qx::HotShape<SHAPE>::kBlock, per = 32 * qx::Lane<V>::N, warps = B / 32;
  const int64_t n_tasks = (a.env_count + per - 1) / per;
  unsigned grid = (unsigned)((n_tasks + warps - 1) / warps);
  if (a.merged) {
    if (h->hot_grid == 0) {
      int per_sm = 0;
      cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, qx::quadx_step_hot_kernel<REF, SHAPE, V, true>, B, 0);
      if (e != cudaSuccess) return e;
      h->hot_grid = h->sm_count * (per_sm > 0 ? per_sm : 1);
    }
    qx::StepArgs am = a;
    am.drainers = (uint32_t)h->hot_grid;
    qx::quadx_step_hot_kernel<REF, SHAPE, V, true><<<grid, B, 0, s>>>(h->dev, am);
    return cudaSuccess;
  }
  if (h->pdl && !stream_is_capturing(s)) {
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(B); lc.dynamicSmemBytes = 0; lc.stream = s;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = &at; lc.numAttrs = 1;
    return cudaLaunchKernelEx(&lc, qx::quadx_step_hot_kernel<REF, SHAPE, V, false>, h->dev, a);
  }
  qx::quadx_step_hot_kernel<REF, SHAPE, V, false><<<grid, B, 0, s>>>(h->dev, a);
  return cudaSuccess;
}
template <int SHAPE, class V>
static cudaError_t launch_hot_one(QxHandle* h, const qx::StepArgs& a, cudaStream_t s) {
  return h->ref_constants ? launch_hot_kernel<true, SHAPE, V>(h, a, s) : launch_hot_kernel<false, SHAPE, V>(h, a, s);
}
template <class V>
static cudaError_t launch_hot_shape(QxHandle* h, const qx::StepArgs& a, cudaStream_t s) {
  switch (h->hot_shape) {
    case 3: return launch_hot_one<3, V>(h, a, s);
    case 4: return launch_hot_one<4, V>(h, a, s);
    case 5: return launch_hot_one<5, V>(h, a, s);
    default: return launch_hot_one<0, V>(h, a, s);
  }
}
// the merged launch applies to a handle as a whole (qx_step_end and qx_done_queue depend on it)
static bool use_merged(const QxHandle* h);
// one agent step of the lean kernel (replaces MODE_STEP_DEFER, or MODE_STEP_INLINE with k = 1 and no auto-reset)
static int launch_hot(QxHandle* h, int mode, qx::StepArgs a, cudaStream_t s) {
  if (a.env_count == 0) { a.env_begin = 0; a.env_count = h->n; }
  a.stream_stores = h->stream_stores;
  a.merged = (mode == qx::MODE_STEP_DEFER && use_merged(h)) ? h->merged : 0;
  a.paired_reset = h->paired_reset;
  if (a.merged) a.queue = h->queue;
  cudaError_t e;
#ifdef QX_EXTRA_SHAPES
  if (h->hot_lanes == 4 && h->hot_shape >= 6) {
    switch (h->hot_shape) {
      case 6: e = launch_hot_one<6, qx::S1>(h, a, s); break;
      case 7: e = launch_hot_one<7, qx::S1>(h, a, s); break;
      case 8: e = launch_hot_one<8, qx::S1>(h, a, s); break;
      default: e = launch_hot_one<9, qx::S1>(h, a, s); break;
    }
  } else
#endif
  if (h->hot_lanes == 2) e = launch_hot_shape<qx::P2<true>>(h, a, s);
  else if (h->hot_lanes == 4) e = launch_hot_shape<qx::S1>(h, a, s);
  else e = launch_hot_shape<float>(h, a, s);
  QX_CUDA(e);
  ++g_launches;
  QX_CUDA(cudaGetLastError());
  return QX_OK;
}
// batches above this size take the lean kernel; QX_HOT=0 / 1 at qx_create forces never / always
constexpr int64_t kHotMinEnvs = 32768;
static bool use_hot(const QxHandle* h) {  // decided per handle, not per launch: a chunked call must run the same arithmetic as a whole one
  if (!h->hot_ok || h->hot_mode == 0) return false;
  return h->hot_mode == 1 || h->n >= kHotMinEnvs;
}
static bool use_merged(const QxHandle* h) { return use_hot(h) && h->cfg.auto_reset && h->merged; }

static int launch(QxHandle* h, int mode, qx::StepArgs a, cudaStream_t s) {
  if (a.env_count == 0) { a.env_begin = 0; a.env_count = h->n; }
  if (use_hot(h) && (mode == qx::MODE_STEP_DEFER || (mode == qx::MODE_STEP_INLINE && a.k == 1 && !h->cfg.auto_reset)))
    return launch_hot(h, mode, a, s);
  if (mode == qx::MODE_RESET_QUEUE && use_hot(h) && h->paired_reset) {
    const unsigned blocks = (unsigned)((a.env_count + 127) / 128);
    const unsigned g = blocks < (unsigned)qx::kResetQueueBlocks ? blocks : (unsigned)qx::kResetQueueBlocks;
    if (h->pdl && !stream_is_capturing(s)) {  // programmatic dependent of the kernel before it on the stream (the step launch in a
                                              // tight loop of qx_step); the kernel waits on the device first
      cudaLaunchConfig_t lc{};
      lc.gridDim = dim3(g); lc.blockDim = dim3(128); lc.dynamicSmemBytes = 0; lc.stream = s;
      cudaLaunchAttribute at{};
      at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at.val.programmaticStreamSerializationAllowed = 1;
      lc.attrs = &at; lc.numAttrs = 1;
      QX_CUDA(h->ref_constants ? cudaLaunchKernelEx(&lc, qx::quadx_reset_hot_kernel<true>, h->dev, a)
                               : cudaLaunchKernelEx(&lc, qx::quadx_reset_hot_kernel<false>, h->dev, a));
    } else if (h->ref_constants) qx::quadx_reset_hot_kernel<true><<<g, 128, 0, s>>>(h->dev, a);
    else qx::quadx_reset_hot_kernel<false><<<g, 128, 0, s>>>(h->dev, a);
    ++g_launches;
    QX_CUDA(cudaGetLastError());
    return QX_OK;
  }
  if (h->dev.task == QX_TASK_YAW) launch_task<QX_TASK_YAW, false, false>(h, mode, a, s);
  else if (h->dev.flight_mode != 0) launch_task<QX_TASK_HOVER, true, false>(h, mode, a, s);
  else if (h->ref_constants) launch_task<QX_TASK_HOVER, false, true>(h, mode, a, s);
  else launch_task<QX_TASK_HOVER, false, false>(h, mode, a, s);
  ++g_launches;
  QX_CUDA(cudaGetLastError());
  return QX_OK;
}

// The kernels access these buffers with vector instructions, which fault on a misaligned address: observation rows are
// written as 16-byte (f32) / 8-byte (bf16) vectors when obs_stride is a multiple of 4 (write_obs; any other stride takes
// the scalar stores), hover actions are read as one float4 per env and terminal-observation rows (stride obs_dim) are
// written as float4.  A call that would issue such an access is refused before anything is launched.
static bool misaligned(const void* p, uintptr_t bytes) { return p && reinterpret_cast<uintptr_t>(p) % bytes != 0; }
static int check_alignment(const QxHandle* h, const char* fn, const float* actions_dev, const void* obs_dev, int32_t obs_dtype,
                           int64_t obs_stride, const float* terminal_obs_dev) {
  if (obs_stride % 4 == 0 && misaligned(obs_dev, obs_dtype == QX_OBS_BF16 ? 8 : 16))
    return fail(QX_EINVAL, "%s: obs_dev must be 16-byte (f32) / 8-byte (bf16) aligned when obs_stride is a multiple of 4", fn);
  if (h->dev.task == QX_TASK_HOVER && misaligned(actions_dev, 16)) return fail(QX_EINVAL, "%s: actions_dev must be 16-byte aligned", fn);
  if (misaligned(terminal_obs_dev, 16)) return fail(QX_EINVAL, "%s: terminal_obs_dev must be 16-byte aligned", fn);
  return QX_OK;
}

extern "C" int qx_reset(QxHandle* h, const uint8_t* mask_dev, void* obs_dev, int32_t obs_dtype, int64_t obs_stride, void* stream) {
  if (!h) return fail(QX_EINVAL, "qx_reset: null handle");
  if (obs_dev && obs_stride < h->dev.obs_dim) return fail(QX_EINVAL, "qx_reset: obs_stride < obs_dim");
  if (int rc = check_alignment(h, "qx_reset", nullptr, obs_dev, obs_dtype, obs_stride, nullptr)) return rc;
  qx::StepArgs a{};
  a.state = h->state; a.mask = mask_dev; a.obs = obs_dev; a.obs_stride = obs_stride; a.obs_bf16 = obs_dtype == QX_OBS_BF16;
  a.stats = h->stats; a.n = h->n; a.k = 1;
  return launch(h, qx::MODE_RESET_MASK, a, (cudaStream_t)stream);
}

extern "C" int qx_step_k(QxHandle* h, int32_t k, const float* actions_dev, float* obs_dev, float* reward_dev,
                         uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream) {
  if (!h || k <= 0 || !actions_dev || !reward_dev || !terminated_dev || !truncated_dev)
    return fail(QX_EINVAL, "qx_step_k: bad arguments");
  if (int rc = check_alignment(h, "qx_step_k", actions_dev, obs_dev, QX_OBS_F32, h->dev.obs_dim, nullptr)) return rc;
  qx::StepArgs a{};
  a.state = h->state; a.actions = actions_dev; a.obs = obs_dev; a.obs_stride = h->dev.obs_dim; a.reward = reward_dev;
  a.terminated = terminated_dev; a.truncated = truncated_dev; a.stats = h->stats; a.n = h->n; a.k = k;
  return launch(h, qx::MODE_STEP_INLINE, a, (cudaStream_t)stream);
}

extern "C" int qx_step_begin(QxHandle* h, const float* actions_dev, void* obs_dev, int32_t obs_dtype, int64_t obs_stride,
                             float* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev, void* stream) {
  if (!h || !actions_dev || !reward_dev || !terminated_dev || !truncated_dev) return fail(QX_EINVAL, "qx_step: bad arguments");
  if (obs_dev && obs_stride < h->dev.obs_dim) return fail(QX_EINVAL, "qx_step: obs_stride < obs_dim");
  if (int rc = check_alignment(h, "qx_step", actions_dev, obs_dev, obs_dtype, obs_stride, terminal_obs_dev)) return rc;
  qx::StepArgs a{};
  a.state = h->state; a.actions = actions_dev; a.obs = obs_dev; a.obs_stride = obs_stride; a.obs_bf16 = obs_dtype == QX_OBS_BF16;
  a.reward = reward_dev; a.terminated = terminated_dev; a.truncated = truncated_dev; a.terminal_obs = terminal_obs_dev;
  a.stats = h->stats; a.n = h->n; a.k = 1;
  if (!h->cfg.auto_reset) return launch(h, qx::MODE_STEP_INLINE, a, (cudaStream_t)stream);
  a.queue = h->queue;
  return launch(h, qx::MODE_STEP_DEFER, a, (cudaStream_t)stream);
}

extern "C" int qx_step_end(QxHandle* h, void* obs_dev, int32_t obs_dtype, int64_t obs_stride, void* stream) {
  if (!h) return fail(QX_EINVAL, "qx_step_end: null handle");
  if (!h->cfg.auto_reset) return QX_OK;
  if (obs_dev && obs_stride < h->dev.obs_dim) return fail(QX_EINVAL, "qx_step_end: obs_stride < obs_dim");
  if (int rc = check_alignment(h, "qx_step_end", nullptr, obs_dev, obs_dtype, obs_stride, nullptr)) return rc;
  if (use_merged(h)) return QX_OK;  // the step launch already re-created the finished envs
  qx::StepArgs a{};
  a.state = h->state; a.obs = obs_dev; a.obs_stride = obs_stride; a.obs_bf16 = obs_dtype == QX_OBS_BF16;
  a.stats = h->stats; a.queue = h->queue; a.n = h->n; a.k = 1;
  return launch(h, qx::MODE_RESET_QUEUE, a, (cudaStream_t)stream);
}

// two launches: the step proper, then the reset of whatever finished, in full warps.  Small batches are latency-bound
// (4 096 envs = one warp per SM sub-partition on 32 SMs), where the second launch costs more than the divergence it
// avoids: below kInlineResetMaxEnvs the finished envs are reset inside the step launch instead.
constexpr int64_t kInlineResetMaxEnvs = 16384;
extern "C" int qx_step(QxHandle* h, const float* actions_dev, void* obs_dev, int32_t obs_dtype, int64_t obs_stride,
                       float* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev, void* stream) {
  if (h && h->cfg.auto_reset && h->n <= kInlineResetMaxEnvs && !(h->hot_mode == 1 && h->hot_ok)) {
    if (!actions_dev || !reward_dev || !terminated_dev || !truncated_dev) return fail(QX_EINVAL, "qx_step: bad arguments");
    if (obs_dev && obs_stride < h->dev.obs_dim) return fail(QX_EINVAL, "qx_step: obs_stride < obs_dim");
    if (int rc = check_alignment(h, "qx_step", actions_dev, obs_dev, obs_dtype, obs_stride, terminal_obs_dev)) return rc;
    qx::StepArgs a{};
    a.state = h->state; a.actions = actions_dev; a.obs = obs_dev; a.obs_stride = obs_stride; a.obs_bf16 = obs_dtype == QX_OBS_BF16;
    a.reward = reward_dev; a.terminated = terminated_dev; a.truncated = truncated_dev; a.terminal_obs = terminal_obs_dev;
    a.stats = h->stats; a.n = h->n; a.k = 1;
    return launch(h, qx::MODE_STEP_INLINE, a, (cudaStream_t)stream);
  }
  int rc = qx_step_begin(h, actions_dev, obs_dev, obs_dtype, obs_stride, reward_dev, terminated_dev, truncated_dev, terminal_obs_dev, stream);
  if (rc) return rc;
  return qx_step_end(h, obs_dev, obs_dtype, obs_stride, stream);
}

// debug hook (not in the public header): out_dev[0] = clock64 of one SM, out_dev[1] = globaltimer ns, enqueued on `stream`
extern "C" int qx_debug_clock_probe(unsigned long long* out_dev, void* stream) {
  if (!out_dev) return fail(QX_EINVAL, "qx_debug_clock_probe: null buffer");
  qx::clock_probe_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(out_dev);
  QX_CUDA(cudaGetLastError());
  return QX_OK;
}

extern "C" int qx_render(QxHandle* h, const int32_t* env_idx_dev, int64_t m, int32_t fmt, uint8_t* frames_dev, void* stream) {
  if (!h) return fail(QX_EINVAL, "qx_render: null handle");
  if (h->dev.task != QX_TASK_HOVER) return fail(QX_EINVAL, "qx_render: camera frames are drawn for the hover task only");
  if (fmt != QX_FRAME_RGBA && fmt != QX_FRAME_MASK) return fail(QX_EINVAL, "qx_render: fmt is QX_FRAME_RGBA or QX_FRAME_MASK");
  if (m < 0) return fail(QX_EINVAL, "qx_render: m < 0");
  if (!env_idx_dev && m != h->n) return fail(QX_EINVAL, "qx_render: env_idx_dev is NULL, so m must equal n_envs");
  const int res = (int)h->cfg.cam_res;
  if (!(h->cfg.cam_res >= 4.f && h->cfg.cam_res <= 8192.f) || (float)res != h->cfg.cam_res || res % 4 != 0)
    return fail(QX_EINVAL, "qx_render: cam_res must be a positive multiple of 4");
  if (!frames_dev && m > 0) return fail(QX_EINVAL, "qx_render: null frames_dev");
  if (reinterpret_cast<uintptr_t>(frames_dev) % 16 != 0) return fail(QX_EINVAL, "qx_render: frames_dev must be 16-byte aligned");
  if (m == 0) return QX_OK;
  qx::RenderArgs a{h->state, h->n, env_idx_dev, m, frames_dev, res, h->raster};
  const int64_t warps = m * ((res + 31) / 32);
  const unsigned grid = (unsigned)((warps + qx::kRenderBlock / 32 - 1) / (qx::kRenderBlock / 32));
  // a plain launch: the step kernels release their programmatic dependents before they store the state planes read here
  if (fmt == QX_FRAME_RGBA) qx::render_kernel<QX_FRAME_RGBA><<<grid, qx::kRenderBlock, 0, (cudaStream_t)stream>>>(a);
  else qx::render_kernel<QX_FRAME_MASK><<<grid, qx::kRenderBlock, 0, (cudaStream_t)stream>>>(a);
  ++g_launches;
  QX_CUDA(cudaGetLastError());
  return QX_OK;
}

extern "C" int qx_episode_record(QxHandle* h, float* ret_dev, int32_t* len_dev, uint32_t* end_dev, uint32_t* n_closed_dev, void* stream) {
  if (!h) return fail(QX_EINVAL, "qx_episode_record: null handle");
  // with auto-reset the reset of a finished env clears its flags word (and its return) before a record could see them
  if (h->cfg.auto_reset) return fail(QX_EINVAL, "qx_episode_record: the handle must be created with auto_reset = 0");
  if (!ret_dev || !len_dev || !end_dev || !n_closed_dev) return fail(QX_EINVAL, "qx_episode_record: null output pointer");
  const unsigned grid = (unsigned)((h->n + qx::kRecordBlock - 1) / qx::kRecordBlock);
  // a plain launch: it starts after the step launch before it has stored the state planes
  qx::episode_record_kernel<<<grid, qx::kRecordBlock, 0, (cudaStream_t)stream>>>(h->state, h->n, ret_dev, len_dev, end_dev, n_closed_dev);
  ++g_launches;
  QX_CUDA(cudaGetLastError());
  return QX_OK;
}

extern "C" int qx_done_queue(QxHandle* h, const uint32_t** count_dev, const uint32_t** idx_dev) {
  if (!h || !count_dev || !idx_dev) return fail(QX_EINVAL, "qx_done_queue: bad arguments");
  *count_dev = &h->queue->published;  // written by the step launch; count itself is zeroed by the reset launch
  *idx_dev = h->queue->idx;
  return QX_OK;
}

static int ensure_staging(QxHandle* h) {
  if (h->staging) return QX_OK;
  const int64_t n = h->n;
  const int od = h->dev.obs_dim, ad = h->dev.act_dim;
  QX_CUDA(cudaMallocHost(&h->h_act, sizeof(float) * n * ad)); QX_CUDA(cudaMalloc(&h->d_act, sizeof(float) * n * ad));
  QX_CUDA(cudaMallocHost(&h->h_obs, sizeof(float) * n * od)); QX_CUDA(cudaMalloc(&h->d_obs, sizeof(float) * n * od));
  QX_CUDA(cudaMallocHost(&h->h_rew, sizeof(float) * n)); QX_CUDA(cudaMalloc(&h->d_rew, sizeof(float) * n));
  QX_CUDA(cudaMallocHost(&h->h_flags, 3 * n)); QX_CUDA(cudaMalloc(&h->d_flags, 3 * n));
  QX_CUDA(cudaMallocHost(&h->h_tobs, sizeof(float) * n * od)); QX_CUDA(cudaMalloc(&h->d_tobs, sizeof(float) * n * od));
  h->staging = true;
  return QX_OK;
}


extern "C" int qx_reset_host(QxHandle* h, const uint8_t* mask_host, float* obs_host) {
  if (!h) return fail(QX_EINVAL, "qx_reset_host: null handle");
  DeviceGuard g(h->device);
  int rc = ensure_staging(h);
  if (rc) return rc;
  const int64_t n = h->n;
  const int od = h->dev.obs_dim;
  uint8_t* dmask = nullptr;
  if (mask_host) {
    memcpy(h->h_flags + 2 * n, mask_host, n);
    QX_CUDA(cudaMemcpyAsync(h->d_flags + 2 * n, h->h_flags + 2 * n, n, cudaMemcpyHostToDevice, h->stream));
    dmask = h->d_flags + 2 * n;
  }
  rc = qx_reset(h, dmask, h->d_obs, QX_OBS_F32, od, h->stream);
  if (rc) return rc;
  if (obs_host) QX_CUDA(cudaMemcpyAsync(h->h_obs, h->d_obs, sizeof(float) * n * od, cudaMemcpyDeviceToHost, h->stream));
  QX_CUDA(cudaStreamSynchronize(h->stream));
  if (obs_host) {
    if (!mask_host) memcpy(obs_host, h->h_obs, sizeof(float) * n * od);
    else
      for (int64_t i = 0; i < n; ++i)
        if (mask_host[i]) memcpy(obs_host + i * od, h->h_obs + i * od, sizeof(float) * od);
  }
  return QX_OK;
}

static bool is_pinned(const void* p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return at.type == cudaMemoryTypeHost;
}

// Pinned caller buffers are used in place; pageable ones go through the handle's pinned staging area.  Large
// batches are cut into chunks and pipelined over three streams -- actions H2D (chunk k+1) | step + reset kernels
// (chunk k) | results D2H (chunk k-1) -- so the PCIe transfers, which dominate this call, overlap the kernels and
// each other (H2D and D2H use different copy engines).
static int step_host_impl(QxHandle* h, const float* actions_host, void* obs_host, const int32_t obs_dtype, float* reward_host,
                          uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host) {
  if (!h || !actions_host) return fail(QX_EINVAL, "qx_step_host: bad arguments");
  if (obs_dtype != QX_OBS_F32 && obs_dtype != QX_OBS_BF16) return fail(QX_EINVAL, "qx_step_host: obs_dtype is QX_OBS_F32 or QX_OBS_BF16");
  const bool bf16 = obs_dtype == QX_OBS_BF16;
  const size_t osz = bf16 ? 2 : 4;  // bytes per observation element on the wire
  DeviceGuard g(h->device);
  int rc = ensure_staging(h);
  if (rc) return rc;
  const int64_t n = h->n;
  const int od = h->dev.obs_dim, ad = h->dev.act_dim;
  const float* src = actions_host;
  if (!is_pinned(actions_host)) { memcpy(h->h_act, actions_host, sizeof(float) * n * ad); src = h->h_act; }
  const bool p_obs = is_pinned(obs_host), p_rew = is_pinned(reward_host), p_te = is_pinned(terminated_host),
             p_tr = is_pinned(truncated_host);
  char* dst_obs = obs_host ? (p_obs ? (char*)obs_host : (char*)h->h_obs) : nullptr;
  float* dst_rew = reward_host ? (p_rew ? reward_host : h->h_rew) : nullptr;
  // the handle's own copy of the flags is only needed to unpack pageable buffers and to pick the terminal observations
  const bool own_flags = terminal_obs_host || (terminated_host && !p_te) || (truncated_host && !p_tr);
  // The D2H engine bounds the call (46 of the 62 bytes per env-step, ~50 GB/s with the H2D running beside it), so (a) it must start
  // early -- the first piece is small: its H2D and kernels are the only time the engine idles -- and (b) it must not stop -- every
  // piece costs ~12 us of gaps between its copies.  Default: five pieces of 1/16, 1/16, 1/8, 1/4, 1/2 of the batch (measured on
  // B200, 1 Mi envs: 9 equal-ish pieces 1.145 ms, 5 pieces 1.10 ms, 3 pieces 1.09 ms).  QX_HOST_CHUNKS = k > 0: k equal pieces, the
  // first one halved again; k < 0: -k geometric pieces (tuning).
  const int nc = h->host_chunks;
  int chunks = 1;
  int64_t begin[17] = {0};
  const int64_t q = 2 * qx::kBlock;  // piece boundaries are multiples of two blocks
  if (n >= (1 << 17)) {
    if (nc > 0) {
      const int64_t per = ((n + nc - 1) / nc + q - 1) / q * q;
      chunks = nc + 1;
      for (int k = 0; k <= chunks; ++k) begin[k] = k == 0 ? 0 : (k == 1 ? per / 2 : (int64_t)(k - 1) * per);
    } else {  // geometric: g pieces of n / 2^(g-1) x (1, 1, 2, 4, ...)
      const int g = nc < 0 ? -nc : 5;
      const int64_t u = ((n >> (g - 1)) + q - 1) / q * q;
      chunks = g;
      for (int k = 1; k < g; ++k) begin[k] = u << (k - 1);
    }
  }
  begin[chunks] = n;
  for (int k = 0; k < chunks; ++k) {
    const int64_t b = begin[k] < n ? begin[k] : n;
    const int64_t e = begin[k + 1] < n ? begin[k + 1] : n;
    const int64_t cnt = e - b;
    if (cnt <= 0) continue;
    QX_CUDA(cudaMemcpyAsync(h->d_act + b * ad, src + b * ad, sizeof(float) * cnt * ad, cudaMemcpyHostToDevice, h->h2d_stream));
    QX_CUDA(cudaEventRecord(h->ev_h2d[k], h->h2d_stream));
    QX_CUDA(cudaStreamWaitEvent(h->stream, h->ev_h2d[k], 0));
    qx::StepArgs a{};
    a.state = h->state; a.actions = h->d_act; a.obs = h->d_obs; a.obs_stride = od; a.obs_bf16 = bf16; a.reward = h->d_rew;
    a.terminated = h->d_flags; a.truncated = h->d_flags + n; a.terminal_obs = terminal_obs_host ? h->d_tobs : nullptr;
    a.stats = h->stats; a.queue = h->queue; a.n = n; a.k = 1; a.env_begin = b; a.env_count = cnt;
    if (h->cfg.auto_reset && (n > kInlineResetMaxEnvs || (h->hot_mode == 1 && h->hot_ok))) {
      rc = launch(h, qx::MODE_STEP_DEFER, a, h->stream);
      if (rc) return rc;
      if (!use_merged(h)) rc = launch(h, qx::MODE_RESET_QUEUE, a, h->stream);
    } else {  // no auto-reset, or a small batch: one launch (see qx_step)
      rc = launch(h, qx::MODE_STEP_INLINE, a, h->stream);
    }
    if (rc) return rc;
    QX_CUDA(cudaEventRecord(h->ev_k[k], h->stream));
    QX_CUDA(cudaStreamWaitEvent(h->d2h_stream, h->ev_k[k], 0));
    QX_CUDA(cudaStreamWaitEvent(h->d2h2_stream, h->ev_k[k], 0));
    if (dst_obs) QX_CUDA(cudaMemcpyAsync(dst_obs + b * od * osz, (const char*)h->d_obs + b * od * osz, osz * cnt * od, cudaMemcpyDeviceToHost, h->d2h_stream));
    cudaStream_t s2 = h->host_one_d2h ? h->d2h_stream : h->d2h2_stream;
    if (dst_rew) QX_CUDA(cudaMemcpyAsync(dst_rew + b, h->d_rew + b, sizeof(float) * cnt, cudaMemcpyDeviceToHost, s2));
    if (own_flags) {
      QX_CUDA(cudaMemcpyAsync(h->h_flags + b, h->d_flags + b, cnt, cudaMemcpyDeviceToHost, s2));
      QX_CUDA(cudaMemcpyAsync(h->h_flags + n + b, h->d_flags + n + b, cnt, cudaMemcpyDeviceToHost, s2));
    }
    if (p_te) QX_CUDA(cudaMemcpyAsync(terminated_host + b, h->d_flags + b, cnt, cudaMemcpyDeviceToHost, s2));
    if (p_tr) QX_CUDA(cudaMemcpyAsync(truncated_host + b, h->d_flags + n + b, cnt, cudaMemcpyDeviceToHost, s2));
  }
  if (terminal_obs_host) QX_CUDA(cudaMemcpyAsync(h->h_tobs, h->d_tobs, sizeof(float) * n * od, cudaMemcpyDeviceToHost, h->d2h_stream));
  QX_CUDA(cudaStreamSynchronize(h->d2h2_stream));
  QX_CUDA(cudaStreamSynchronize(h->d2h_stream));
  QX_CUDA(cudaStreamSynchronize(h->stream));
  if (obs_host && !p_obs) memcpy(obs_host, h->h_obs, osz * n * od);
  if (reward_host && !p_rew) memcpy(reward_host, h->h_rew, sizeof(float) * n);
  if (terminated_host && !p_te) memcpy(terminated_host, h->h_flags, n);
  if (truncated_host && !p_tr) memcpy(truncated_host, h->h_flags + n, n);
  if (terminal_obs_host) {
    for (int64_t i = 0; i < n; ++i)
      if (h->h_flags[i] || h->h_flags[n + i]) memcpy(terminal_obs_host + i * od, h->h_tobs + i * od, sizeof(float) * od);
  }
  return QX_OK;
}

extern "C" int qx_step_host(QxHandle* h, const float* actions_host, float* obs_host, float* reward_host,
                            uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host) {
  return step_host_impl(h, actions_host, obs_host, QX_OBS_F32, reward_host, terminated_host, truncated_host, terminal_obs_host);
}

extern "C" int qx_step_host_ex(QxHandle* h, const float* actions_host, void* obs_host, int32_t obs_dtype, float* reward_host,
                               uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host) {
  return step_host_impl(h, actions_host, obs_host, obs_dtype, reward_host, terminated_host, truncated_host, terminal_obs_host);
}

extern "C" int qx_get_state(QxHandle* h, void* planes_host) {
  if (!h || !planes_host) return fail(QX_EINVAL, "qx_get_state: bad arguments");
  DeviceGuard g(h->device);
  // device layout: h->planes planes of n float4; host layout: 4 * h->planes planes of n words
  const int64_t n = h->n;
  const int P = h->planes;
  float4* tmp = (float4*)malloc(sizeof(float4) * P * n);
  if (!tmp) return fail(QX_ENOMEM, "qx_get_state: out of host memory");
  cudaError_t e = cudaMemcpy(tmp, h->state, sizeof(float4) * P * n, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) { free(tmp); return fail(QX_ECUDA, "qx_get_state: %s", cudaGetErrorString(e)); }
  float* out = (float*)planes_host;
  for (int p = 0; p < P; ++p)
    for (int64_t i = 0; i < n; ++i) {
      const float4 v = tmp[p * n + i];
      out[(4 * p + 0) * n + i] = v.x; out[(4 * p + 1) * n + i] = v.y; out[(4 * p + 2) * n + i] = v.z; out[(4 * p + 3) * n + i] = v.w;
    }
  free(tmp);
  return QX_OK;
}

// the flags word (QX_FLAG_*) of envs [first, first + count): a strided copy of one word per env, no full-state transfer
extern "C" int qx_get_flags(QxHandle* h, int64_t first, int64_t count, uint32_t* flags_host) {
  if (!h || !flags_host || first < 0 || count <= 0 || first + count > h->n) return fail(QX_EINVAL, "qx_get_flags: bad arguments");
  DeviceGuard g(h->device);
  const float4* plane = h->state + 7 * h->n + first;  // plane 7 = (svb2, step_count, rng_ctr, flags)
  QX_CUDA(cudaMemcpy2D(flags_host, sizeof(uint32_t), reinterpret_cast<const char*>(plane) + 12, sizeof(float4), sizeof(uint32_t), (size_t)count,
                       cudaMemcpyDeviceToHost));
  return QX_OK;
}

extern "C" int qx_set_state(QxHandle* h, const void* planes_host) {
  if (!h || !planes_host) return fail(QX_EINVAL, "qx_set_state: bad arguments");
  DeviceGuard g(h->device);
  const int64_t n = h->n;
  const int P = h->planes;
  float4* tmp = (float4*)malloc(sizeof(float4) * P * n);
  if (!tmp) return fail(QX_ENOMEM, "qx_set_state: out of host memory");
  const float* in = (const float*)planes_host;
  for (int p = 0; p < P; ++p)
    for (int64_t i = 0; i < n; ++i)
      tmp[p * n + i] = make_float4(in[(4 * p + 0) * n + i], in[(4 * p + 1) * n + i], in[(4 * p + 2) * n + i], in[(4 * p + 3) * n + i]);
  cudaError_t e = cudaMemcpy(h->state, tmp, sizeof(float4) * P * n, cudaMemcpyHostToDevice);
  free(tmp);
  if (e != cudaSuccess) return fail(QX_ECUDA, "qx_set_state: %s", cudaGetErrorString(e));
  return QX_OK;
}

extern "C" int qx_episode_stats(QxHandle* h, double* sum_return, int64_t* sum_length, int64_t* n_episodes, int32_t clear) {
  if (!h) return fail(QX_EINVAL, "qx_episode_stats: null handle");
  DeviceGuard g(h->device);
  qx::Stats s;
  QX_CUDA(cudaMemcpy(&s, h->stats, sizeof(s), cudaMemcpyDeviceToHost));
  if (clear) QX_CUDA(cudaMemset(h->stats, 0, offsetof(qx::Stats, n_nonfinite)));  // the failure counter is since creation
  if (sum_return) *sum_return = s.sum_ret;
  if (sum_length) *sum_length = (int64_t)s.sum_len;
  if (n_episodes) *n_episodes = (int64_t)s.n_done;
  return QX_OK;
}
