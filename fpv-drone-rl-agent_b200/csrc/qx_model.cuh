// qx_model.cuh -- fp32 device model of one QuadX drone + the hover / yaw env layer.
//
// Everything here runs in registers of ONE thread per env.  What is computed
// follows, step by step,
//   * /root/reference/simulation/hover.py:224-358 (obs, reward, termination, step)
//   * hover.py:72-113 (reset), yaw.py:57-149 (yaw task)
//   * the PyFlyt 0.21.0 QuadX model (mode 0, plus the outer loops of modes -1..7) and pybullet's multibody integrator
//     as restated in SURVEY.md section 9 (third-party, parity unpinned),
//     parameterised by cf2x.yaml:1-54 and cf2x.urdf:10-68.
// It is written from that description for this hardware, not translated from
// the CPU oracle: single precision, MUFU intrinsics, no libm slow paths inside
// the sub-step loop, Philox counters instead of a stateful generator.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "qx_lanes.cuh"

namespace qx {

// ---------------------------------------------------------------------------
// kernel-side constants, derived once on the host from QxConfig
// ---------------------------------------------------------------------------
struct DevConfig {
  int32_t task, n_sub_step, n_sub_reset, ctrl_every, max_steps, floor_grace, render, auto_reset, noise,
      state_stale, gyro, obs_dim, act_dim;
  float h, lag_alpha, one_m_alpha, noise_ratio, noise_k, thrust_k, pwm_idle;  // noise_k = -2 ln2 noise_ratio^2
  float torque_k[4], mx[4], my[4], map[16];
  float drag_c, drag_pqr, kp[3], kiT[3], kd_T[3], lim[3];
  float inv_mass, g, I[3], invI[3], vmax, floor_z;
  float hI[3], hm, hg, hh, hh2, ndrag_c, ndrag_pqr, kq1, kq2;  // h/I, h/m, h g, h/2, (h/2)^2, -drag, series coefficients * h/2
  float gk[3];                                                 // gyroscopic term: -(h / I_k) (I_(k+2) - I_(k+1)), or 0 when off
  float cam_sd, cam_cd, inv_tan, res, half_res, inv_half_res, inv_res2, cam_near, cam_off[3], margin, panel[12];
  float inv_agent_dt, dome2, floor_thr, target_area, target_ratio, act_scale[3];
  float start_pos[3], start_rpy[3], spawn_thr, spawn_pos_noise, spawn_yaw_noise;
  uint32_t seed_lo, seed_hi, env_lo, env_hi;  // env id of local env 0
  // PyFlyt flight modes (cascade instantiation only): outer-loop gains as kp[w] ki*T[w] kd/T[w] lim[w]
  int32_t flight_mode, need_euler;
  float thrust_scale, thrust_bias;
  float att[12], vel[8], lpos[8], zpos[4], zvel[4];
  // motor geometry folded with the thrust scale: torque_x = sum arm_y[m] rr[m], torque_y = sum arm_x[m] rr[m]
  // (arm_x = -thrust_k mx, arm_y = thrust_k my).  x_layout: the four props sit on a symmetric X (cf2x.urdf:35-68) with
  // torque signs (-,-,+,+), so the sums share partial sums (arm_k = thrust_k |mx|, tq_k = torque_k[2]); x_mixer: the
  // motor map is the +-1 matrix of that layout, so the mixer is eight adds.
  int32_t x_layout, x_mixer;
  float arm_x[4], arm_y[4], arm_k, tq_k;
  // camera features: 0 = analytic projection of the front face (vision()), 1 = scan conversion of the box silhouette
  // on the pixel lattice (vision_raster()); panel_back = the four corners of the face behind panel[]
  int32_t vision_mode;
  const float* raster;  // vision_mode 1: 36 floats in device memory (RasterConsts), written by qx_create
};

}  // namespace qx
// The reference's own parameter set (hover.py / cf2x.yaml / cf2x.urdf literals) as compile-time constants: a second
// instantiation of the step kernel overwrites the model fields of its DevConfig copy with these literals, so they
// become immediates instead of ~33 constant-bank loads per Aviary.step and a few dozen live registers.  It is selected
// at qx_create only when derive() produced exactly these bits; any other configuration runs the generic kernel.
#include "qx_ref_constants.cuh"
namespace qx {

enum : uint32_t {
  F_CONTACT = 1u,
  F_TERM = 2u,
  F_TRUNC = 4u,
  F_OOB = 8u,
  F_ONFLOOR = 16u,
  F_LOWZ = 32u,
};
enum : uint32_t { STREAM_STEP = 0, STREAM_RESET = 1, STREAM_SPAWN = 2 };

// What the physics sub-steps and the rate controller read and write, for one env (T = float) or two (T = float2).
template <class T>
struct Core {
  T px, py, pz;           // world position
  T qx, qy, qz, qw;       // body->world quaternion (x,y,z,w)
  T vx, vy, vz;           // world linear velocity
  T wx, wy, wz;           // BODY-frame angular velocity (see physics_substep)
  T thr[4];               // motor throttle (PyFlyt Motors.throttle)
  T pi[3], pe[3];         // rate PID integral, previous error
  T swb[3], svb[3];       // Aviary.state rows 0 and 2 (body rates / velocity snapshot)
  typename Lane<T>::mask contact;  // resting on the floor stand-in (F_CONTACT of the stored flags word)
  // transient (not stored): pose part of the Aviary.state snapshot
  T sqx, sqy, sqz, sqw, spx, spy, spz;
};

// The 44 carried words of one env (QX_STATE_WORDS); plane p, lane l = word 4p+l.  Planes 0..7 are what the sub-step
// loop needs (Core + counters + flags), planes 8..10 only the once-per-step epilogue -- the two-env kernel loads those
// after the loop, so they do not occupy registers across it.
struct Env : Core<float> {
  int32_t step_count;         // hover.py:356
  uint32_t rng_ctr;           // env steps since creation (Philox counter word 2)
  uint32_t flags;
  float peul[3];              // previous_ang_pos, hover.py:354
  float ep_ret;               // Monitor: running episode return
  float pa[4];                // prev_action, hover.py:357
  float pcx, pcy, parea, pratio;  // hover.py:270-272
  // cascade instantiation only (planes 11..16; spx/spy/spz are carried there too): (integral, previous error) of
  // ang_pos 0/3, lin_vel 6/8, lin_pos 10/12, z_vel 14/15, z_pos 16/17
  float cp[18];
};

// NC: the read-only path (ld.global.nc) -- only where no thread of the same launch wrote the word before; the reset phase
// of the merged step kernel re-reads planes its own launch stored and takes the L2-coherent path instead.
template <bool NC = true> QX_DI float4 ldg4(const float4* p) { return NC ? __ldg(p) : __ldcg(p); }

constexpr int kLoopPlanes = 8;  // planes 0..7: sub-step loop state
QX_DI void unpack_loop_planes(Env& e, const float4 (&v)[kLoopPlanes]) {
  e.px = v[0].x; e.py = v[0].y; e.pz = v[0].z; e.qx = v[0].w;
  e.qy = v[1].x; e.qz = v[1].y; e.qw = v[1].z; e.vx = v[1].w;
  e.vy = v[2].x; e.vz = v[2].y; e.wx = v[2].z; e.wy = v[2].w;
  e.wz = v[3].x; e.thr[0] = v[3].y; e.thr[1] = v[3].z; e.thr[2] = v[3].w;
  e.thr[3] = v[4].x; e.pi[0] = v[4].y; e.pi[1] = v[4].z; e.pi[2] = v[4].w;
  e.pe[0] = v[5].x; e.pe[1] = v[5].y; e.pe[2] = v[5].z; e.swb[0] = v[5].w;
  e.swb[1] = v[6].x; e.swb[2] = v[6].y; e.svb[0] = v[6].z; e.svb[1] = v[6].w;
  e.svb[2] = v[7].x; e.step_count = __float_as_int(v[7].y); e.rng_ctr = __float_as_uint(v[7].z); e.flags = __float_as_uint(v[7].w);
  e.contact = (e.flags & F_CONTACT) != 0u;
  e.sqx = e.qx; e.sqy = e.qy; e.sqz = e.qz; e.sqw = e.qw; e.spx = e.px; e.spy = e.py; e.spz = e.pz;
}
template <bool NC = true>
QX_DI void load_env_loop(Env& e, const float4* __restrict__ st, int64_t n, int64_t i) {
  float4 v[kLoopPlanes];
#pragma unroll
  for (int p = 0; p < kLoopPlanes; ++p) v[p] = ldg4<NC>(st + (int64_t)p * n + i);
  unpack_loop_planes(e, v);
}
QX_DI void unpack_tail_planes(Env& e, const float4 k, const float4 l, const float4 m) {
  e.peul[0] = k.x; e.peul[1] = k.y; e.peul[2] = k.z; e.ep_ret = k.w;
  e.pa[0] = l.x; e.pa[1] = l.y; e.pa[2] = l.z; e.pa[3] = l.w;
  e.pcx = m.x; e.pcy = m.y; e.parea = m.z; e.pratio = m.w;
}
template <bool NC = true>
QX_DI void load_env_tail(Env& e, const float4* __restrict__ st, int64_t n, int64_t i) {
  unpack_tail_planes(e, ldg4<NC>(st + 8 * n + i), ldg4<NC>(st + 9 * n + i), ldg4<NC>(st + 10 * n + i));
}
template <bool NC = true>
QX_DI void load_env(Env& e, const float4* __restrict__ st, int64_t n, int64_t i) {
  load_env_loop<NC>(e, st, n, i);
  load_env_tail<NC>(e, st, n, i);
}

template <bool CS = false>
QX_DI void store_env(const Env& e, float4* __restrict__ st, int64_t n, int64_t i) {
  const uint32_t flags = (e.flags & ~F_CONTACT) | (e.contact ? F_CONTACT : 0u);
  auto put = [&](int p, float4 v) {
    if (CS) __stcs(st + (int64_t)p * n + i, v);
    else st[(int64_t)p * n + i] = v;
  };
  put(0, make_float4(e.px, e.py, e.pz, e.qx));
  put(1, make_float4(e.qy, e.qz, e.qw, e.vx));
  put(2, make_float4(e.vy, e.vz, e.wx, e.wy));
  put(3, make_float4(e.wz, e.thr[0], e.thr[1], e.thr[2]));
  put(4, make_float4(e.thr[3], e.pi[0], e.pi[1], e.pi[2]));
  put(5, make_float4(e.pe[0], e.pe[1], e.pe[2], e.swb[0]));
  put(6, make_float4(e.swb[1], e.swb[2], e.svb[0], e.svb[1]));
  put(7, make_float4(e.svb[2], __int_as_float(e.step_count), __uint_as_float(e.rng_ctr), __uint_as_float(flags)));
  put(8, make_float4(e.peul[0], e.peul[1], e.peul[2], e.ep_ret));
  put(9, make_float4(e.pa[0], e.pa[1], e.pa[2], e.pa[3]));
  put(10, make_float4(e.pcx, e.pcy, e.parea, e.pratio));
}

// Flight modes != 0: six more planes -- the outer loops' PID memory and the position row of the Aviary.state
// snapshot, which those loops read at the first control update of the next step.
constexpr int kBasePlanes = 11, kCascadePlanes = 17;
QX_DI void load_cascade(Env& e, const float4* __restrict__ st, int64_t n, int64_t i) {
  float4 v[6];
#pragma unroll
  for (int p = 0; p < 6; ++p) v[p] = ldg4(st + (int64_t)(kBasePlanes + p) * n + i);
  const float* w = reinterpret_cast<const float*>(v);
#pragma unroll
  for (int k = 0; k < 18; ++k) e.cp[k] = w[k];
  e.spx = w[18]; e.spy = w[19]; e.spz = w[20];
}
QX_DI void store_cascade(const Env& e, float4* __restrict__ st, int64_t n, int64_t i) {
  st[(int64_t)(kBasePlanes + 0) * n + i] = make_float4(e.cp[0], e.cp[1], e.cp[2], e.cp[3]);
  st[(int64_t)(kBasePlanes + 1) * n + i] = make_float4(e.cp[4], e.cp[5], e.cp[6], e.cp[7]);
  st[(int64_t)(kBasePlanes + 2) * n + i] = make_float4(e.cp[8], e.cp[9], e.cp[10], e.cp[11]);
  st[(int64_t)(kBasePlanes + 3) * n + i] = make_float4(e.cp[12], e.cp[13], e.cp[14], e.cp[15]);
  st[(int64_t)(kBasePlanes + 4) * n + i] = make_float4(e.cp[16], e.cp[17], e.spx, e.spy);
  st[(int64_t)(kBasePlanes + 5) * n + i] = make_float4(e.spz, 0.f, 0.f, 0.f);
}

// two scalar envs <-> one two-lane Core (register renaming only)
template <class P>
QX_DI void pack_core(Core<P>& p, const Core<float>& a, const Core<float>& b) {
#define mk2(u, v) P{u, v}
  p.px = mk2(a.px, b.px); p.py = mk2(a.py, b.py); p.pz = mk2(a.pz, b.pz);
  p.qx = mk2(a.qx, b.qx); p.qy = mk2(a.qy, b.qy); p.qz = mk2(a.qz, b.qz); p.qw = mk2(a.qw, b.qw);
  p.vx = mk2(a.vx, b.vx); p.vy = mk2(a.vy, b.vy); p.vz = mk2(a.vz, b.vz);
  p.wx = mk2(a.wx, b.wx); p.wy = mk2(a.wy, b.wy); p.wz = mk2(a.wz, b.wz);
#pragma unroll
  for (int m = 0; m < 4; ++m) p.thr[m] = mk2(a.thr[m], b.thr[m]);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    p.pi[k] = mk2(a.pi[k], b.pi[k]); p.pe[k] = mk2(a.pe[k], b.pe[k]);
    p.swb[k] = mk2(a.swb[k], b.swb[k]); p.svb[k] = mk2(a.svb[k], b.svb[k]);
  }
  p.contact = m2{a.contact, b.contact};
  p.sqx = mk2(a.sqx, b.sqx); p.sqy = mk2(a.sqy, b.sqy); p.sqz = mk2(a.sqz, b.sqz); p.sqw = mk2(a.sqw, b.sqw);
  p.spx = mk2(a.spx, b.spx); p.spy = mk2(a.spy, b.spy); p.spz = mk2(a.spz, b.spz);
#undef mk2
}
template <int HALF, class P>
QX_DI void unpack_core(Core<float>& a, const Core<P>& p) {
#define QX_H(v) (HALF ? (v).y : (v).x)
  a.px = QX_H(p.px); a.py = QX_H(p.py); a.pz = QX_H(p.pz);
  a.qx = QX_H(p.qx); a.qy = QX_H(p.qy); a.qz = QX_H(p.qz); a.qw = QX_H(p.qw);
  a.vx = QX_H(p.vx); a.vy = QX_H(p.vy); a.vz = QX_H(p.vz);
  a.wx = QX_H(p.wx); a.wy = QX_H(p.wy); a.wz = QX_H(p.wz);
#pragma unroll
  for (int m = 0; m < 4; ++m) a.thr[m] = QX_H(p.thr[m]);
#pragma unroll
  for (int k = 0; k < 3; ++k) { a.pi[k] = QX_H(p.pi[k]); a.pe[k] = QX_H(p.pe[k]); a.swb[k] = QX_H(p.swb[k]); a.svb[k] = QX_H(p.svb[k]); }
  a.contact = HALF ? p.contact.y : p.contact.x;
  a.sqx = QX_H(p.sqx); a.sqy = QX_H(p.sqy); a.sqz = QX_H(p.sqz); a.sqw = QX_H(p.sqw);
  a.spx = QX_H(p.spx); a.spy = QX_H(p.spy); a.spz = QX_H(p.spz);
#undef QX_H
}

// ---------------------------------------------------------------------------
// Philox4x32-R: same integer stream as oracle/quadx_model.py:philox4x32.  The env's motor / spawn noise uses R = 7
// (Random123: the smallest round count that passes BigCrush); the policy's action sampling keeps R = 10.
// ---------------------------------------------------------------------------
constexpr int kEnvPhiloxRounds = 7;
template <int ROUNDS>
QX_DI uint4 philox4x32(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}
QX_DI uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) { return philox4x32<10>(c, k0, k1); }
QX_DI uint4 env_philox(uint4 c, uint32_t k0, uint32_t k1) { return philox4x32<kEnvPhiloxRounds>(c, k0, k1); }

// ((x >> 9) + 0.5) * 2^-23 without an int->float conversion (reset pose noise)
QX_DI float u01(uint32_t x) { return __uint_as_float((x >> 9) | 0x3f800000u) - 0.99999994f; }
// the 16-bit halves of a word as floats k in [0, 65535] (one I2F.U16 each: the conversion takes the half-word operand directly,
// where building 1 + k 2^-16 in the mantissa costs a shift, a mask and an or per field)
QX_DI float f16_lo16(uint32_t w) { return __uint2float_rn(w & 0xffffu); }
QX_DI float f16_hi16(uint32_t w) { return __uint2float_rn(w >> 16); }
template <class T> QX_DI T f16_lo(uint32_t w) { return f16_lo16(w); }
template <class T> QX_DI T f16_hi(uint32_t w) { return f16_hi16(w); }
template <class T> QX_DI T f16_lo(uint2 w) { return T{f16_lo16(w.x), f16_lo16(w.y)}; }
template <class T> QX_DI T f16_hi(uint2 w) { return T{f16_hi16(w.x), f16_hi16(w.y)}; }
// Box-Muller inputs from a field k: u = (k + 0.5) 2^-16 in (0,1), angle = 2 pi u - pi.  Written on m = 1 + k 2^-16 these were
// u = m - (1 - 2^-17) and angle = fma(m, c, -d) with c = 6.28318530718f, d = 9.42473002f; on k they are the same real numbers
// rounded once -- u is exact either way, and c - d is exactly representable, so fma(k, c 2^-16, c - d) == fma(m, c, -d) bit for bit
// (oracle/quadx_model.py:normal4 and oracle/quadx_oracle.c keep the m form; tests/test_gpu_parity.py compares the streams).
constexpr float kBmU0 = 7.62939453125e-06f, kBmUk = 1.52587890625e-05f;             // 2^-17, 2^-16
constexpr float kBmTk = 6.28318530718f * 1.52587890625e-05f, kBmT0 = 6.28318530718f - 9.42473002f;

// 4 x noise_ratio * N(0,1) from two 32-bit words, like oracle normal4(): each word is one Box-Muller pair
// (low half -> radius, high half -> angle).  u = m - (1 - 2^-17) = (k + 0.5) 2^-16 in (0,1);  the scale is folded into
// the radius: noise_ratio sqrt(-2 ln u) = sqrt(noise_k lg2 u);  the angle is 2 pi u - pi in (-pi, pi), where the MUFU
// sine / cosine are most accurate, = 2 pi m - (2 pi (1 - 2^-17) + pi).
template <class T, class U>
QX_DI void normal4_scaled(U w0, U w1, float noise_k, T n[4]) {
  const T ra = vsqrt(vmul(vlg2(vfma(f16_lo<T>(w0), kBmUk, splat<T>(kBmU0))), noise_k));
  const T rb = vsqrt(vmul(vlg2(vfma(f16_lo<T>(w1), kBmUk, splat<T>(kBmU0))), noise_k));
  const T ta = vfma(f16_hi<T>(w0), kBmTk, splat<T>(kBmT0));
  const T tb = vfma(f16_hi<T>(w1), kBmTk, splat<T>(kBmT0));
  n[0] = vmul(ra, vcos(ta)); n[1] = vmul(ra, vsin(ta)); n[2] = vmul(rb, vcos(tb)); n[3] = vmul(rb, vsin(tb));
}

// ---------------------------------------------------------------------------
// PyFlyt QuadX.update_control, mode 0: rate PID -> motor mix -> saturation
// ---------------------------------------------------------------------------
// apwm[] returns lag_alpha * pwm: the motor lag thr += alpha (pwm - thr) is applied as thr (1 - alpha) + (alpha pwm)
template <class T>
QX_DI void control_update(Core<T>& e, const DevConfig& c, const T sp[4], T apwm[4]) {
  T cmd[4], pwm[4];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const T err = vsub(sp[a], e.swb[a]);
    e.pi[a] = vclamp(vfma(err, c.kiT[a], e.pi[a]), -c.lim[a], c.lim[a]);
    T u = vfma(err, c.kp[a], e.pi[a]);
    if (c.kd_T[a] != 0.f) u = vfma(vsub(err, e.pe[a]), c.kd_T[a], u);
    cmd[a] = vclamp(u, -c.lim[a], c.lim[a]);
    e.pe[a] = err;
  }
  cmd[3] = sp[3];
  if (c.x_mixer) {  // rows (-,-,-,+) (+,+,-,+) (+,-,+,+) (-,+,+,+): shared sums and differences
    const T s = vadd(cmd[0], cmd[1]), d = vsub(cmd[0], cmd[1]), a = vsub(cmd[3], cmd[2]), b = vadd(cmd[3], cmd[2]);
    pwm[0] = vsub(a, s); pwm[1] = vadd(a, s); pwm[2] = vadd(b, d); pwm[3] = vsub(b, d);
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m)
      pwm[m] = vfma(cmd[3], c.map[4 * m + 3], vfma(cmd[2], c.map[4 * m + 2], vfma(cmd[1], c.map[4 * m + 1], vmul(cmd[0], c.map[4 * m + 0]))));
  }
  const T high = vmax(vmax(pwm[0], pwm[1]), vmax(pwm[2], pwm[3]));
  const auto over = vgt(high, 1.0f);
  if (vany(over)) {
    const T inv = vsel(over, vrcp(high), 1.0f);
#pragma unroll
    for (int m = 0; m < 4; ++m) pwm[m] = vmul(pwm[m], inv);
  }
  const T low = vmin(vmin(pwm[0], pwm[1]), vmin(pwm[2], pwm[3]));
  const auto under = vlt(low, c.pwm_idle);
  if (vany(under)) {
    const T k = vsel(under, vmul(vsub(c.pwm_idle, low), vrcp(vsub(1.0f, low))), 0.f);
#pragma unroll
    for (int m = 0; m < 4; ++m) pwm[m] = vfma(vsub(1.0f, pwm[m]), k, pwm[m]);
  }
#pragma unroll
  for (int m = 0; m < 4; ++m) apwm[m] = vmul(pwm[m], c.lag_alpha);
}

// ---------------------------------------------------------------------------
// PyFlyt PID.step for one channel; g = kp[w] ki*T[w] kd/T[w] lim[w], channel k
// ---------------------------------------------------------------------------
template <int W>
QX_DI float pid_channel(const float* g, int k, float& mi, float& me, float state, float sp) {
  const float err = sp - state, lim = g[3 * W + k];
  mi = clampf(fmaf(g[W + k], err, mi), -lim, lim);
  const float d = g[2 * W + k] * (err - me);
  me = err;
  return clampf(fmaf(g[k], err, mi) + d, -lim, lim);
}

// QuadX.update_control for flight modes != 0: the outer loops turn the setpoint into (rate commands, thrust) and the
// mode-0 controller above finishes the job.  seul = Euler row of the Aviary.state snapshot.  Mode -1 bypasses
// everything (setpoint = motor pwm, no mixing, no saturation).
QX_DI void control_update_cascade(Env& e, const DevConfig& c, const float sp[4], const float seul[3], float pwm[4]) {
  const int mode = c.flight_mode;
  if (mode == -1) {
#pragma unroll
    for (int m = 0; m < 4; ++m) pwm[m] = sp[m] * c.lag_alpha;
    return;
  }
  float a[4] = {sp[0], sp[1], sp[2], sp[3]};
  if (mode == 1 || mode == 3) {  // angles -> rates
#pragma unroll
    for (int k = 0; k < 3; ++k) a[k] = pid_channel<3>(c.att, k, e.cp[k], e.cp[3 + k], seul[k], a[k]);
  } else if (mode >= 4) {
    if (mode == 7) {  // ground-frame position -> ground-frame velocity
      a[0] = pid_channel<2>(c.lpos, 0, e.cp[10], e.cp[12], e.spx, a[0]);
      a[1] = pid_channel<2>(c.lpos, 1, e.cp[11], e.cp[13], e.spy, a[1]);
    }
    if (mode >= 6) {  // ground frame -> yaw-rotated local frame
      float sy, cy;
      sincosf(seul[2], &sy, &cy);
      const float gx = a[0], gy = a[1];
      a[0] = cy * gx + sy * gy;
      a[1] = cy * gy - sy * gx;
    }
    // local velocity -> tilt angles: +x needs +pitch, +y needs -roll
    const float ang0 = pid_channel<2>(c.vel, 0, e.cp[6], e.cp[8], e.svb[0], a[0]);
    const float ang1 = pid_channel<2>(c.vel, 1, e.cp[7], e.cp[9], e.svb[1], a[1]);
    a[0] = -ang1; a[1] = ang0;
    a[0] = pid_channel<3>(c.att, 0, e.cp[0], e.cp[3], seul[0], a[0]);
    a[1] = pid_channel<3>(c.att, 1, e.cp[1], e.cp[4], seul[1], a[1]);
    if (mode == 7) a[2] = pid_channel<3>(c.att, 2, e.cp[2], e.cp[5], seul[2], a[2]);  // yaw is an angle only in mode 7
  }
  if (mode == 2 || mode == 3 || mode == 4 || mode == 7) a[3] = pid_channel<1>(c.zpos, 0, e.cp[16], e.cp[17], e.spz, a[3]);
  if (mode != 0) a[3] = pid_channel<1>(c.zvel, 0, e.cp[14], e.cp[15], e.svb[2], a[3]);
  a[3] = __saturatef(a[3]);
  control_update<float>(e, c, a, pwm);
}

// ---------------------------------------------------------------------------
// one 1/physics_hz sub-step: Motors.physics_update + drag + update_state +
// pybullet.stepSimulation (free flight) + the declared floor stand-in.
//
// Bullet integrates the WORLD angular velocity, w' = w + h R a_b, and then
// q' = exp(h w'/2) q.  With w = R w_b that is exactly  w_b' = w_b + h a_b  and
// q' = q exp(h w_b'/2)  (a rotation about u leaves u unchanged), so the
// angular half is carried in the body frame and needs no rotation matrix.
// (Bullet's +-100 clamp acts on world components; here on body components --
// the two differ only beyond 100 rad/s.)
// ---------------------------------------------------------------------------
// cold path: an env at or below the floor plane -- sticky plane at floor_z (zeroes world v_xy and world w_xy)
template <class T, class M>
QX_DI void floor_contact(Core<T>& e, const DevConfig& c, const M below) {
  e.pz = vsel(below, c.floor_z, e.pz);
  e.vz = vsel(below, vmax(e.vz, splat<T>(0.f)), e.vz);
  e.vx = vsel(below, 0.f, e.vx);
  e.vy = vsel(below, 0.f, e.vy);
  const T X = e.qx, Y = e.qy, Z = e.qz, W = e.qw;
  const T a20 = vmul(vsub(vmul(X, Z), vmul(W, Y)), 2.f), a21 = vmul(vfma(Y, Z, vmul(W, X)), 2.f);
  const T a22 = vsub(1.f, vmul(vfma(X, X, vmul(Y, Y)), 2.f));
  const T wzw = vfma(a22, e.wz, vfma(a21, e.wy, vmul(a20, e.wx)));  // world yaw rate survives
  e.wx = vsel(below, vmul(a20, wzw), e.wx);
  e.wy = vsel(below, vmul(a21, wzw), e.wy);
  e.wz = vsel(below, vmul(a22, wzw), e.wz);
}

template <class T>
QX_DI void physics_substep(Core<T>& e, const DevConfig& c, const T apwm[4], const T nz[4], const bool last) {
  // motors: first-order lag, multiplicative noise, thrust and torques
  T rr[4];
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    T t = vfma(e.thr[m], c.one_m_alpha, apwm[m]);
    t = vfma(nz[m], t, t);                // nz already scaled by noise_ratio
    e.thr[m] = t;
    rr[m] = vabsmul(t, t);                // rpm |rpm| / max_rpm^2
  }
  T fz, tx, ty, tz;                       // r x F = (y F, -x F, 0)
  if (c.x_layout) {  // sums and differences of the motor pairs (0,2) and (1,3): the order the pair-packed kernel uses
    const T s0 = vadd(rr[0], rr[2]), s1 = vadd(rr[1], rr[3]), d0 = vsub(rr[0], rr[2]), d1 = vsub(rr[1], rr[3]);
    fz = vadd(s0, s1);
    tx = vmul(vsub(d1, d0), c.arm_k); ty = vmul(vsub(s1, s0), c.arm_k); tz = vmul(vadd(d0, d1), -c.tq_k);
  } else {
    fz = vadd(vadd(rr[0], rr[1]), vadd(rr[2], rr[3]));
    tx = vmul(rr[0], c.arm_y[0]); ty = vmul(rr[0], c.arm_x[0]); tz = vmul(rr[0], c.torque_k[0]);
#pragma unroll
    for (int m = 1; m < 4; ++m) { tx = vfma(rr[m], c.arm_y[m], tx); ty = vfma(rr[m], c.arm_x[m], ty); tz = vfma(rr[m], c.torque_k[m], tz); }
  }
  if (c.thrust_k != 1.0f) fz = vmul(fz, c.thrust_k);
  // drag from the (stale) snapshot, body frame
  const T fbx = vmul(vabsmul(e.svb[0], c.ndrag_c), e.svb[0]);
  const T fby = vmul(vabsmul(e.svb[1], c.ndrag_c), e.svb[1]);
  const T fbz = vfma(vabsmul(e.svb[2], c.ndrag_c), e.svb[2], fz);
  if (vany(e.contact)) {  // no angular drag while resting on the floor (cold)
    const T dq = vsel(e.contact, splat<T>(0.f), c.ndrag_pqr);
    tx = vfma(vabsmul(e.swb[0], dq), e.swb[0], tx);
    ty = vfma(vabsmul(e.swb[1], dq), e.swb[1], ty);
    tz = vfma(vabsmul(e.swb[2], dq), e.swb[2], tz);
  } else {
    tx = vfma(vabsmul(e.swb[0], c.ndrag_pqr), e.swb[0], tx);
    ty = vfma(vabsmul(e.swb[1], c.ndrag_pqr), e.swb[1], ty);
    tz = vfma(vabsmul(e.swb[2], c.ndrag_pqr), e.swb[2], tz);
  }
  // rotation matrix of the current attitude
  const T x = e.qx, y = e.qy, z = e.qz, w = e.qw;
  const T x2 = vadd(x, x), y2 = vadd(y, y), z2 = vadd(z, z);
  const T wx = vmul(w, x2), wy = vmul(w, y2), wz = vmul(w, z2);
  const Neg<T> nx2 = mkneg(x2), ny2 = mkneg(y2), nz2 = mkneg(z2), nwx = mkneg(wx), nwy = mkneg(wy), nwz = mkneg(wz);
  const T r00 = vfnma(y, ny2, vfnma1(z, nz2)), r11 = vfnma(x, nx2, vfnma1(z, nz2)), r22 = vfnma(x, nx2, vfnma1(y, ny2));
  const T r01 = vfms(x, y2, nwz), r10 = vfma(x, y2, wz);
  const T r02 = vfma(x, z2, wy), r20 = vfms(x, z2, nwy);
  const T r12 = vfms(y, z2, nwx), r21 = vfma(y, z2, wx);
  if (c.state_stale) {  // QuadX.update_state runs before stepSimulation
    e.swb[0] = e.wx; e.swb[1] = e.wy; e.swb[2] = e.wz;
    e.svb[0] = vfma(r20, e.vz, vfma(r10, e.vy, vmul(r00, e.vx)));
    e.svb[1] = vfma(r21, e.vz, vfma(r11, e.vy, vmul(r01, e.vx)));
    e.svb[2] = vfma(r22, e.vz, vfma(r12, e.vy, vmul(r02, e.vx)));
    if (last) { e.sqx = x; e.sqy = y; e.sqz = z; e.sqw = w; e.spx = e.px; e.spy = e.py; e.spz = e.pz; }  // only the final pose is read
  }
  // angular half, body frame
  // w x (I w) for a diagonal inertia is ((I2 - I1) wy wz, (I0 - I2) wz wx, (I1 - I0) wx wy); gk = -h / I_k times those
  // differences (0 when the gyroscopic term is off), so each axis is one product and two FFMA
  const T wyz = vmul(e.wy, e.wz), wzx = vmul(e.wz, e.wx), wxy = vmul(e.wx, e.wy);
  e.wx = vfma(wyz, c.gk[0], vfma(tx, c.hI[0], e.wx));
  e.wy = vfma(wzx, c.gk[1], vfma(ty, c.hI[1], e.wy));
  e.wz = c.gk[2] != 0.f ? vfma(wxy, c.gk[2], vfma(tz, c.hI[2], e.wz)) : vfma(tz, c.hI[2], e.wz);
  // linear half, world frame: semi-implicit Euler
  e.vx = vfma(vfma(r02, fbz, vfma(r01, fby, vmul(r00, fbx))), c.hm, e.vx);
  e.vy = vfma(vfma(r12, fbz, vfma(r11, fby, vmul(r10, fbx))), c.hm, e.vy);
  e.vz = vadd(vfma(vfma(r22, fbz, vfma(r21, fby, vmul(r20, fbx))), c.hm, e.vz), -c.hg);
  // btMultiBody's +-max_coord_vel clamp: one max over the six components, the clamp itself is a cold path
  if (vany(vgt(vmax(vmax(vabsmax(e.vx, e.vy), vabsmax(e.vz, e.wx)), vabsmax(e.wy, e.wz)), c.vmax))) {
    e.vx = vclamp(e.vx, -c.vmax, c.vmax); e.vy = vclamp(e.vy, -c.vmax, c.vmax); e.vz = vclamp(e.vz, -c.vmax, c.vmax);
    e.wx = vclamp(e.wx, -c.vmax, c.vmax); e.wy = vclamp(e.wy, -c.vmax, c.vmax); e.wz = vclamp(e.wz, -c.vmax, c.vmax);
  }
  e.px = vfma(e.vx, c.h, e.px);
  e.py = vfma(e.vy, c.h, e.py);
  e.pz = vfma(e.vz, c.h, e.pz);
  // q <- q exp(h w_b / 2): series in s = (|w| h / 2)^2 (no sqrt / sin / cos), then renormalise
  // sin(x)/x * h/2 and cos(x) in s = x^2, x = |w| h / 2 <= 0.37 at the +-100 rad/s clamp: truncation < 4e-9
  // The product is formed as q + q (dq - 1): the increment is ~|w| h / 2 relative to q, so its rounding is negligible and
  // each component takes one rounding at |q| scale instead of one per FFMA of the full product -- the attitude random
  // walk over thousands of sub-steps is what drives the open-loop position drift against the float64 oracle.
  const T s = vmul(vfma(e.wz, e.wz, vfma(e.wy, e.wy, vmul(e.wx, e.wx))), c.hh2);
  const T kq = vfma(s, vfma(s, c.kq2, c.kq1), c.hh);
  const T dwm1 = vmul(s, vfma(s, vfma(s, -1.f / 720.f, 1.f / 24.f), -0.5f));  // cos(|w| h / 2) - 1
  const T dx = vmul(e.wx, kq), dy = vmul(e.wy, kq), dz = vmul(e.wz, kq);
  const Neg<T> ndx = mkneg(dx), ndy = mkneg(dy), ndz = mkneg(dz);
  // (term order chosen so that (nx, ny) and (nz, nw) are each one chain of pair operations in the pair-packed kernel)
  const T nx = vadd(x, vfnma(z, ndy, vfma(y, dz, vfma(x, dwm1, vmul(w, dx)))));
  const T ny = vadd(y, vfma(z, dx, vfnma(x, ndz, vfma(y, dwm1, vmul(w, dy)))));
  const T nzq = vadd(z, vfnma(y, ndx, vfma(x, dy, vfma(z, dwm1, vmul(w, dz)))));
  const T nw = vadd(w, vfnma(y, ndy, vfnma(x, ndx, vfnma(z, ndz, vmul(w, dwm1)))));
  const T inv = vrsqrt(vadd(vfma(nzq, nzq, vmul(nx, nx)), vfma(nw, nw, vmul(ny, ny))));
  e.qx = vmul(nx, inv); e.qy = vmul(ny, inv); e.qz = vmul(nzq, inv); e.qw = vmul(nw, inv);
  // floor stand-in
  const auto below = vlt(e.pz, c.floor_z);
  if (vany(below)) floor_contact(e, c, below);  // (ptxas if-converts this block; a warp-uniform VOTE + branch around it measured 2 % slower)
  e.contact = below;
  if (!c.state_stale) {
    const T X = e.qx, Y = e.qy, Z = e.qz, W = e.qw;
    const T X2 = vadd(X, X), Y2 = vadd(Y, Y), Z2 = vadd(Z, Z);
    const T a00 = vsub(1.f, vfma(Y2, Y, vmul(Z2, Z))), a01 = vsub(vmul(X, Y2), vmul(W, Z2)), a02 = vfma(X, Z2, vmul(W, Y2));
    const T a10 = vfma(X, Y2, vmul(W, Z2)), a11 = vsub(1.f, vfma(X2, X, vmul(Z2, Z))), a12 = vsub(vmul(Y, Z2), vmul(W, X2));
    const T a20 = vsub(vmul(X, Z2), vmul(W, Y2)), a21 = vfma(Y, Z2, vmul(W, X2)), a22 = vsub(1.f, vfma(X2, X, vmul(Y2, Y)));
    e.swb[0] = e.wx; e.swb[1] = e.wy; e.swb[2] = e.wz;
    e.svb[0] = vfma(a20, e.vz, vfma(a10, e.vy, vmul(a00, e.vx)));
    e.svb[1] = vfma(a21, e.vz, vfma(a11, e.vy, vmul(a01, e.vx)));
    e.svb[2] = vfma(a22, e.vz, vfma(a12, e.vy, vmul(a02, e.vx)));
    if (last) { e.sqx = X; e.sqy = Y; e.sqz = Z; e.sqw = W; e.spx = e.px; e.spy = e.py; e.spz = e.pz; }
  }
}

// ===========================================================================
// The same sub-step for ONE env with its own components paired: (x, y) of every vector, motors (0, 1) and (2, 3) and
// (z, w) of the quaternion sit in aligned register pairs, so that the component-wise arithmetic issues as packed
// FFMA2 / FMUL2 / FADD2 (one issue slot for two components; the FMA pipe is busy for two cycles either way, but issue
// slots are what bound this kernel).  Every component goes through the same IEEE operations in the same order as in
// physics_substep<float> / control_update<float> above, so the two are bitwise identical -- with one precondition:
// motor throttles are never negative (|t| t == t t), which holds for flight mode 0 with spawn_throttle >= 0 and
// pwm_idle >= 0 (qx_create checks it before it selects this code).
// ===========================================================================
struct S1 {};  // lane tag: one env per thread, its own components paired
template <> struct Lane<S1> { typedef bool mask; typedef uint32_t u32; static constexpr int N = 1; };
struct CoreS {
  f2 pxy, qxy, qzw, vxy, wxy, thr01, thr23, pixy, pexy, swbxy;
  float pz, vz, wz, piz, pez, swbz, svb[3];
  bool contact;
  float sqx, sqy, sqz, sqw, spx, spy, spz;  // transient: pose part of the Aviary.state snapshot
};
QX_DI void pack_core_s(CoreS& p, const Core<float>& a) {
  p.pxy = f2{a.px, a.py}; p.pz = a.pz; p.qxy = f2{a.qx, a.qy}; p.qzw = f2{a.qz, a.qw};
  p.vxy = f2{a.vx, a.vy}; p.vz = a.vz; p.wxy = f2{a.wx, a.wy}; p.wz = a.wz;
  p.thr01 = f2{a.thr[0], a.thr[1]}; p.thr23 = f2{a.thr[2], a.thr[3]};
  p.pixy = f2{a.pi[0], a.pi[1]}; p.piz = a.pi[2]; p.pexy = f2{a.pe[0], a.pe[1]}; p.pez = a.pe[2];
  p.swbxy = f2{a.swb[0], a.swb[1]}; p.swbz = a.swb[2];
  p.svb[0] = a.svb[0]; p.svb[1] = a.svb[1]; p.svb[2] = a.svb[2];
  p.contact = a.contact;
  p.sqx = a.sqx; p.sqy = a.sqy; p.sqz = a.sqz; p.sqw = a.sqw; p.spx = a.spx; p.spy = a.spy; p.spz = a.spz;
}
QX_DI void unpack_core_s(Core<float>& a, const CoreS& p) {
  a.px = p.pxy.x; a.py = p.pxy.y; a.pz = p.pz; a.qx = p.qxy.x; a.qy = p.qxy.y; a.qz = p.qzw.x; a.qw = p.qzw.y;
  a.vx = p.vxy.x; a.vy = p.vxy.y; a.vz = p.vz; a.wx = p.wxy.x; a.wy = p.wxy.y; a.wz = p.wz;
  a.thr[0] = p.thr01.x; a.thr[1] = p.thr01.y; a.thr[2] = p.thr23.x; a.thr[3] = p.thr23.y;
  a.pi[0] = p.pixy.x; a.pi[1] = p.pixy.y; a.pi[2] = p.piz; a.pe[0] = p.pexy.x; a.pe[1] = p.pexy.y; a.pe[2] = p.pez;
  a.swb[0] = p.swbxy.x; a.swb[1] = p.swbxy.y; a.swb[2] = p.swbz;
  a.svb[0] = p.svb[0]; a.svb[1] = p.svb[1]; a.svb[2] = p.svb[2];
  a.contact = p.contact;
  a.sqx = p.sqx; a.sqy = p.sqy; a.sqz = p.sqz; a.sqw = p.sqw; a.spx = p.spx; a.spy = p.spy; a.spz = p.spz;
}
// a pair of config constants: when both halves are the same value ptxas uses the broadcast / immediate operand form
QX_DI f2 cpair(float a, float b) { return f2{a, b}; }

// 4 x noise_ratio N(0,1) of one env as two pairs (n0, n1), (n2, n3): normal4_scaled<float> with the two Box-Muller words paired
QX_DI void normal4_scaled_s(uint32_t w0, uint32_t w1, float noise_k, f2 n[2]) {
  const f2 u = vfma(f2{f16_lo16(w0), f16_lo16(w1)}, kBmUk, f2{kBmU0, kBmU0});
  const f2 t = vfma(f2{f16_hi16(w0), f16_hi16(w1)}, kBmTk, f2{kBmT0, kBmT0});
  const f2 r2 = vmul(f2{__log2f(u.x), __log2f(u.y)}, noise_k);
  const float ra = fsqrt(r2.x), rb = fsqrt(r2.y);
  n[0] = vmul(f2{__cosf(t.x), __sinf(t.x)}, ra);
  n[1] = vmul(f2{__cosf(t.y), __sinf(t.y)}, rb);
}

// control_update<float>, roll / pitch as one pair; spxy = rate setpoints (roll, pitch), spz = yaw rate, thrust = sp[3]
QX_DI void control_update_s(CoreS& e, const DevConfig& c, const f2 spxy, const float spz, const float thrust, f2 apwm[2]) {
  const f2 err = vsub(spxy, e.swbxy);
  f2 pi = vfma(err, cpair(c.kiT[0], c.kiT[1]), e.pixy);
  pi = f2{clampf(pi.x, -c.lim[0], c.lim[0]), clampf(pi.y, -c.lim[1], c.lim[1])};
  e.pixy = pi;
  f2 u = vfma(err, cpair(c.kp[0], c.kp[1]), pi);
  if (c.kd_T[0] != 0.f || c.kd_T[1] != 0.f) {
    const f2 ud = vfma(vsub(err, e.pexy), cpair(c.kd_T[0], c.kd_T[1]), u);
    u = f2{c.kd_T[0] != 0.f ? ud.x : u.x, c.kd_T[1] != 0.f ? ud.y : u.y};
  }
  e.pexy = err;
  const float cmd0 = clampf(u.x, -c.lim[0], c.lim[0]), cmd1 = clampf(u.y, -c.lim[1], c.lim[1]);
  const float errz = spz - e.swbz;
  e.piz = clampf(fmaf(errz, c.kiT[2], e.piz), -c.lim[2], c.lim[2]);
  float uz = fmaf(errz, c.kp[2], e.piz);
  if (c.kd_T[2] != 0.f) uz = fmaf(errz - e.pez, c.kd_T[2], uz);
  const float cmd2 = clampf(uz, -c.lim[2], c.lim[2]);
  e.pez = errz;
  float pwm[4];
  if (c.x_mixer) {  // rows (-,-,-,+) (+,+,-,+) (+,-,+,+) (-,+,+,+): shared sums and differences
    const float s = __fadd_rn(cmd0, cmd1), d = __fsub_rn(cmd0, cmd1), a = __fsub_rn(thrust, cmd2), b = __fadd_rn(thrust, cmd2);
    pwm[0] = __fsub_rn(a, s); pwm[1] = __fadd_rn(a, s); pwm[2] = __fadd_rn(b, d); pwm[3] = __fsub_rn(b, d);
  } else {
#pragma unroll
    for (int m = 0; m < 4; ++m)
      pwm[m] = fmaf(thrust, c.map[4 * m + 3], fmaf(cmd2, c.map[4 * m + 2], fmaf(cmd1, c.map[4 * m + 1], __fmul_rn(cmd0, c.map[4 * m + 0]))));
  }
  const float high = fmaxf(fmaxf(pwm[0], pwm[1]), fmaxf(pwm[2], pwm[3]));
  if (high > 1.0f) {
    const float inv = frcp(high);
#pragma unroll
    for (int m = 0; m < 4; ++m) pwm[m] = __fmul_rn(pwm[m], inv);
  }
  const float low = fminf(fminf(pwm[0], pwm[1]), fminf(pwm[2], pwm[3]));
  if (low < c.pwm_idle) {
    const float k = __fmul_rn(__fsub_rn(c.pwm_idle, low), frcp(__fsub_rn(1.0f, low)));
#pragma unroll
    for (int m = 0; m < 4; ++m) pwm[m] = fmaf(__fsub_rn(1.0f, pwm[m]), k, pwm[m]);
  }
  apwm[0] = vmul(f2{pwm[0], pwm[1]}, c.lag_alpha);
  apwm[1] = vmul(f2{pwm[2], pwm[3]}, c.lag_alpha);
}

// FLOOR = false: the speculative variant for an env that is not resting on the floor and is expected to stay clear of it --
// the floor stand-in (~24 predicated instructions per sub-step, issued by every warp) is replaced by one FMNMX that tracks the
// lowest pz; the caller re-runs the step with FLOOR = true when that dips below floor_z.  Until it does the two variants go
// through the same operations, so a step that passes the check is bitwise what FLOOR = true computes.
template <bool FLOOR = true>
QX_DI void physics_substep_s(CoreS& e, const DevConfig& c, const f2 apwm[2], const f2 nz[2], const bool last, float& minz) {
  // motors: first-order lag, multiplicative noise, thrust and torques
  f2 t01 = vfma(e.thr01, c.one_m_alpha, apwm[0]), t23 = vfma(e.thr23, c.one_m_alpha, apwm[1]);
  t01 = vfma(nz[0], t01, t01); t23 = vfma(nz[1], t23, t23);
  e.thr01 = t01; e.thr23 = t23;
  const f2 rr01 = vmul(t01, t01), rr23 = vmul(t23, t23);  // throttle >= 0 (see above): |t| t == t t
  float fz, tx, ty, tz;
  if (c.x_layout) {
    const f2 s = vadd(rr01, rr23), d = vsub(rr01, rr23);
    fz = __fadd_rn(s.x, s.y);
    const f2 txy = vmul(f2{__fsub_rn(d.y, d.x), __fsub_rn(s.y, s.x)}, c.arm_k);
    tx = txy.x; ty = txy.y; tz = __fmul_rn(__fadd_rn(d.x, d.y), -c.tq_k);
  } else {
    const float rr[4] = {rr01.x, rr01.y, rr23.x, rr23.y};
    fz = __fadd_rn(__fadd_rn(rr[0], rr[1]), __fadd_rn(rr[2], rr[3]));
    tx = __fmul_rn(rr[0], c.arm_y[0]); ty = __fmul_rn(rr[0], c.arm_x[0]); tz = __fmul_rn(rr[0], c.torque_k[0]);
#pragma unroll
    for (int m = 1; m < 4; ++m) { tx = fmaf(rr[m], c.arm_y[m], tx); ty = fmaf(rr[m], c.arm_x[m], ty); tz = fmaf(rr[m], c.torque_k[m], tz); }
  }
  if (c.thrust_k != 1.0f) fz = __fmul_rn(fz, c.thrust_k);
  // drag from the (stale) snapshot, body frame (|v| does not pack: scalar)
  const float fbx = __fmul_rn(vabsmul(e.svb[0], c.ndrag_c), e.svb[0]);
  const float fby = __fmul_rn(vabsmul(e.svb[1], c.ndrag_c), e.svb[1]);
  const float fbz = fmaf(vabsmul(e.svb[2], c.ndrag_c), e.svb[2], fz);
  {
    const float dq = (FLOOR && e.contact) ? 0.f : c.ndrag_pqr;  // no angular drag while resting on the floor
    tx = fmaf(vabsmul(e.swbxy.x, dq), e.swbxy.x, tx);
    ty = fmaf(vabsmul(e.swbxy.y, dq), e.swbxy.y, ty);
    tz = fmaf(vabsmul(e.swbz, dq), e.swbz, tz);
  }
  // rotation matrix of the current attitude
  const float x = e.qxy.x, y = e.qxy.y, z = e.qzw.x, w = e.qzw.y;
  const f2 xy2 = vadd(e.qxy, e.qxy);
  const float x2 = xy2.x, y2 = xy2.y, z2 = __fadd_rn(z, z);
  const f2 wxy2 = vmul(xy2, w);
  const float wx = wxy2.x, wy = wxy2.y, wz = __fmul_rn(w, z2);
  const float r00 = fmaf(-y, y2, fmaf(-z, z2, 1.f)), r11 = fmaf(-x, x2, fmaf(-z, z2, 1.f)), r22 = fmaf(-x, x2, fmaf(-y, y2, 1.f));
  const float r01 = fmaf(x, y2, -wz), r10 = fmaf(x, y2, wz);
  const float r02 = fmaf(x, z2, wy), r20 = fmaf(x, z2, -wy);
  const float r12 = fmaf(y, z2, -wx), r21 = fmaf(y, z2, wx);
  if (c.state_stale) {  // QuadX.update_state runs before stepSimulation
    e.swbxy = e.wxy; e.swbz = e.wz;
    const float vx = e.vxy.x, vy = e.vxy.y;
    e.svb[0] = fmaf(r20, e.vz, fmaf(r10, vy, __fmul_rn(r00, vx)));
    e.svb[1] = fmaf(r21, e.vz, fmaf(r11, vy, __fmul_rn(r01, vx)));
    e.svb[2] = fmaf(r22, e.vz, fmaf(r12, vy, __fmul_rn(r02, vx)));
    if (last) { e.sqx = x; e.sqy = y; e.sqz = z; e.sqw = w; e.spx = e.pxy.x; e.spy = e.pxy.y; e.spz = e.pz; }
  }
  // angular half, body frame: (wx, wy) as a pair
  {
    const float owx = e.wxy.x, owy = e.wxy.y, owz = e.wz;
    const f2 g = f2{__fmul_rn(owy, owz), __fmul_rn(owz, owx)};
    e.wxy = vfma(g, cpair(c.gk[0], c.gk[1]), vfma(f2{tx, ty}, cpair(c.hI[0], c.hI[1]), e.wxy));
    e.wz = c.gk[2] != 0.f ? fmaf(__fmul_rn(owx, owy), c.gk[2], fmaf(tz, c.hI[2], owz)) : fmaf(tz, c.hI[2], owz);
  }
  // linear half, world frame: (vx, vy) as a pair over the column pairs of R
  {
    const f2 acc = vfma(f2{r02, r12}, fbz, vfma(f2{r01, r11}, fby, vmul(f2{r00, r10}, fbx)));
    e.vxy = vfma(acc, c.hm, e.vxy);
    e.vz = __fadd_rn(fmaf(fmaf(r22, fbz, fmaf(r21, fby, __fmul_rn(r20, fbx))), c.hm, e.vz), -c.hg);
  }
  if (fmaxf(fmaxf(vabsmax(e.vxy.x, e.vxy.y), vabsmax(e.vz, e.wxy.x)), vabsmax(e.wxy.y, e.wz)) > c.vmax) {  // cold
    e.vxy = f2{clampf(e.vxy.x, -c.vmax, c.vmax), clampf(e.vxy.y, -c.vmax, c.vmax)}; e.vz = clampf(e.vz, -c.vmax, c.vmax);
    e.wxy = f2{clampf(e.wxy.x, -c.vmax, c.vmax), clampf(e.wxy.y, -c.vmax, c.vmax)}; e.wz = clampf(e.wz, -c.vmax, c.vmax);
  }
  e.pxy = vfma(e.vxy, c.h, e.pxy);
  e.pz = fmaf(e.vz, c.h, e.pz);
  // q <- q exp(h w_b / 2), then renormalise (same series as physics_substep)
  {
    const float nwx = e.wxy.x, nwy = e.wxy.y, nwz = e.wz;
    const float s = __fmul_rn(fmaf(nwz, nwz, fmaf(nwy, nwy, __fmul_rn(nwx, nwx))), c.hh2);
    const float kq = fmaf(s, fmaf(s, c.kq2, c.kq1), c.hh);
    const float dwm1 = __fmul_rn(s, fmaf(s, fmaf(s, -1.f / 720.f, 1.f / 24.f), -0.5f));
    const f2 dxy = vmul(e.wxy, kq);
    const float dz = __fmul_rn(nwz, kq);
    const f2 jq = f2{y, -x}, jd = f2{-dxy.y, dxy.x};
    // (nx, ny) = (x, y) + w (dx, dy) + dwm1 (x, y) + dz (y, -x) + z (-dy, dx)
    const f2 nxy = vadd(e.qxy, vfma(jd, z, vfma(jq, dz, vfma(e.qxy, dwm1, vmul(dxy, w)))));
    // (nz, nw) = (z, w) + w (dz, dwm1) + z (dwm1, -dz) + (-x) (-dy, dx) + (-y) (dx, dy)
    const f2 nzw = vadd(e.qzw, vfma(dxy, -y, vfma(jd, jq.y, vfma(f2{dwm1, -dz}, z, vmul(f2{dz, dwm1}, w)))));
    const f2 m = vfma(nzw, nzw, vmul(nxy, nxy));
    const float inv = frsqrt(__fadd_rn(m.x, m.y));
    e.qxy = vmul(nxy, inv); e.qzw = vmul(nzw, inv);
  }
  // floor stand-in (cold)
  if constexpr (FLOOR) {
    const bool below = e.pz < c.floor_z;
    if (below) {  // if-converted by ptxas (~24 predicated instructions per sub-step); a VOTE + uniform branch around it measured 2 % slower
      e.pz = c.floor_z; e.vz = fmaxf(e.vz, 0.f); e.vxy = f2{0.f, 0.f};
      const float X = e.qxy.x, Y = e.qxy.y, Z = e.qzw.x, W = e.qzw.y;
      const float a20 = __fmul_rn(__fsub_rn(__fmul_rn(X, Z), __fmul_rn(W, Y)), 2.f), a21 = __fmul_rn(fmaf(Y, Z, __fmul_rn(W, X)), 2.f);
      const float a22 = __fsub_rn(1.f, __fmul_rn(fmaf(X, X, __fmul_rn(Y, Y)), 2.f));
      const float wzw = fmaf(a22, e.wz, fmaf(a21, e.wxy.y, __fmul_rn(a20, e.wxy.x)));  // world yaw rate survives
      e.wxy = f2{__fmul_rn(a20, wzw), __fmul_rn(a21, wzw)}; e.wz = __fmul_rn(a22, wzw);
    }
    e.contact = below;
  } else {
    minz = fminf(minz, e.pz);  // pz < floor_z in any sub-step <=> min pz < floor_z (a NaN pz fails both tests alike)
  }
  if (!c.state_stale) {
    const float X = e.qxy.x, Y = e.qxy.y, Z = e.qzw.x, W = e.qzw.y;
    const float X2 = X + X, Y2 = Y + Y, Z2 = Z + Z;
    const float a00 = __fsub_rn(1.f, fmaf(Y2, Y, __fmul_rn(Z2, Z))), a01 = __fsub_rn(__fmul_rn(X, Y2), __fmul_rn(W, Z2)), a02 = fmaf(X, Z2, __fmul_rn(W, Y2));
    const float a10 = fmaf(X, Y2, __fmul_rn(W, Z2)), a11 = __fsub_rn(1.f, fmaf(X2, X, __fmul_rn(Z2, Z))), a12 = __fsub_rn(__fmul_rn(Y, Z2), __fmul_rn(W, X2));
    const float a20 = __fsub_rn(__fmul_rn(X, Z2), __fmul_rn(W, Y2)), a21 = fmaf(Y, Z2, __fmul_rn(W, X2)), a22 = __fsub_rn(1.f, fmaf(X2, X, __fmul_rn(Y2, Y)));
    e.swbxy = e.wxy; e.swbz = e.wz;
    e.svb[0] = fmaf(a20, e.vz, fmaf(a10, e.vxy.y, __fmul_rn(a00, e.vxy.x)));
    e.svb[1] = fmaf(a21, e.vz, fmaf(a11, e.vxy.y, __fmul_rn(a01, e.vxy.x)));
    e.svb[2] = fmaf(a22, e.vz, fmaf(a12, e.vxy.y, __fmul_rn(a02, e.vxy.x)));
    if (last) { e.sqx = X; e.sqy = Y; e.sqz = Z; e.sqw = W; e.spx = e.pxy.x; e.spy = e.pxy.y; e.spz = e.pz; }
  }
}

// atan2 for finite arguments that are not both zero: octant reduction to t = min / max in [0, 1], t P(t^2) with the degree-7
// minimax P (tools/fit_atan.py: max error 1.2e-7 in fp32 arithmetic, the size of one rounding at pi), ~22 instructions against
// libm's ~50.  The Euler angles are differenced over agent_dt = 1/40 s in the observation: 2.4e-7 rad -> 1e-5 rad/s.
QX_DI float fast_atan2f(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(fmaxf(ax, ay), 1e-30f), mn = fminf(ax, ay);
  const float t = mn * frcp(mx), u = t * t;
  float p = fmaf(u, -0.0040544066578149796f, 0.021862365305423737f);
  p = fmaf(u, p, -0.05591144412755966f);
  p = fmaf(u, p, 0.09642129391431808f);
  p = fmaf(u, p, -0.13908600807189941f);
  p = fmaf(u, p, 0.1994655877351761f);
  p = fmaf(u, p, -0.33329859375953674f);
  p = fmaf(u, p, 0.9999993443489075f);
  float r = t * p;
  r = ay > ax ? 1.57079632679f - r : r;
  r = x < 0.f ? 3.14159265359f - r : r;
  return copysignf(r, y);
}

// pybullet.getEulerFromQuaternion (ZYX, with its gimbal guard)
__device__ __forceinline__ void quat_to_euler(float x, float y, float z, float w, float& roll, float& pitch, float& yaw) {
  const float sarg = -2.f * (x * z - w * y);
  if (sarg <= -0.99999f) {
    roll = 0.f; pitch = -1.57079632679f; yaw = 2.f * atan2f(x, -y);
  } else if (sarg >= 0.99999f) {
    roll = 0.f; pitch = 1.57079632679f; yaw = 2.f * atan2f(-x, y);
  } else {
    roll = fast_atan2f(2.f * (y * z + w * x), w * w - x * x - y * y + z * z);
    pitch = asinf(sarg);
    yaw = fast_atan2f(2.f * (x * y + w * z), w * w + x * x - y * y - z * z);
  }
}

// pybullet.getQuaternionFromEuler, hover.py:233
__device__ __forceinline__ void euler_to_quat(float roll, float pitch, float yaw, float& x, float& y, float& z, float& w) {
  float sr, cr, sp, cp, sy, cy;
  __sincosf(0.5f * roll, &sr, &cr);
  __sincosf(0.5f * pitch, &sp, &cp);
  __sincosf(0.5f * yaw, &sy, &cy);
  x = sr * cp * cy - cr * sp * sy;
  y = cr * sp * cy + sr * cp * sy;
  z = cr * cp * sy - sr * sp * cy;
  w = cr * cp * cy + sr * sp * sy;
}

// ---------------------------------------------------------------------------
// Camera: analytic stand-in for Camera.capture_image + detect_rectangle
// (hover.py:157-222, 241-248).  The four corners of the red face are projected
// through the PyFlyt FPV camera (body Euler angles with the pitch offset by the
// tilt; FOV 90, 128x128) and the features are taken on the pixel lattice the
// way cv2.findContours / contourArea / boundingRect would report them.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void vision(const Env& e, const DevConfig& c, bool& vis, float& cx, float& cy, float& area,
                                       float& ratio) {
  // (every multiply-add is written as fmaf: the library is built with -fmad=false, a * b + c * d would issue three instructions)
  const float x = e.qx, y = e.qy, z = e.qz, w = e.qw;
  const float x2 = x + x, y2 = y + y, z2 = z + z;
  const float wx = w * x2, wy = w * y2, wz = w * z2;
  const float r00 = fmaf(-y, y2, fmaf(-z, z2, 1.f)), r11 = fmaf(-x, x2, fmaf(-z, z2, 1.f)), r22 = fmaf(-x, x2, fmaf(-y, y2, 1.f));
  const float r01 = fmaf(x, y2, -wz), r10 = fmaf(x, y2, wz);
  const float r02 = fmaf(x, z2, wy), r20 = fmaf(x, z2, -wy);
  const float r12 = fmaf(y, z2, -wx), r21 = fmaf(y, z2, wx);
  // sin / cos of the roll Euler angle = (r21, r22) / cos(pitch)
  float sph = 0.f, cph = 1.f;
  if (fabsf(r20) < 0.99999f) {
    const float inv = frsqrt(fmaf(r21, r21, r22 * r22));
    sph = r21 * inv; cph = r22 * inv;
  }
  // camera axes in the body frame: Rx(-roll) Ry(-tilt) Rx(roll) applied to x, z
  const float sd = c.cam_sd, cd = c.cam_cd;
  const float fx = cd, fy = sd * sph, fzz = sd * cph;
  const float ux = -sd * cph, uy = sph * cph * (cd - 1.f), uz = fmaf(sph, sph, cd * cph * cph);
  // right = fwd x up
  const float rx = fmaf(fy, uz, -(fzz * uy)), ry = fmaf(fzz, ux, -(fx * uz)), rz = fmaf(fx, uy, -(fy * ux));
  float pxs[4], pys[4];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float dx = c.panel[3 * k + 0] - e.px, dy = c.panel[3 * k + 1] - e.py, dz = c.panel[3 * k + 2] - e.pz;
    const float bx = fmaf(r20, dz, fmaf(r10, dy, fmaf(r00, dx, -c.cam_off[0])));
    const float by = fmaf(r21, dz, fmaf(r11, dy, fmaf(r01, dx, -c.cam_off[1])));
    const float bz = fmaf(r22, dz, fmaf(r12, dy, fmaf(r02, dx, -c.cam_off[2])));
    const float depth = fmaf(fzz, bz, fmaf(fy, by, fx * bx));
    ok = ok && (depth > c.cam_near);
    const float k1 = c.inv_tan * c.half_res * frcp(fmaxf(depth, 1e-9f));
    pxs[k] = fmaf(fmaf(rz, bz, fmaf(ry, by, rx * bx)), k1, c.half_res);
    pys[k] = fmaf(fmaf(uz, bz, fmaf(uy, by, ux * bx)), -k1, c.half_res);
  }
  const float xmin = fminf(fminf(pxs[0], pxs[1]), fminf(pxs[2], pxs[3]));
  const float xmax = fmaxf(fmaxf(pxs[0], pxs[1]), fmaxf(pxs[2], pxs[3]));
  const float ymin = fminf(fminf(pys[0], pys[1]), fminf(pys[2], pys[3]));
  const float ymax = fmaxf(fmaxf(pys[0], pys[1]), fmaxf(pys[2], pys[3]));
  ok = ok && xmin >= c.margin && ymin >= c.margin && xmax <= c.res - c.margin && ymax <= c.res - c.margin;
  float a2 = 0.f, per = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int kn = (k + 1) & 3;
    a2 += fmaf(pxs[k], pys[kn], -(pxs[kn] * pys[k]));
    const float ex = pxs[kn] - pxs[k], ey = pys[kn] - pys[k];
    per += fsqrt(fmaf(ex, ex, ey * ey));
  }
  const float wpx = floorf(xmax - 0.5f) - ceilf(xmin - 0.5f) + 1.f;
  const float hpx = floorf(ymax - 0.5f) - ceilf(ymin - 0.5f) + 1.f;
  ok = ok && wpx >= 2.f && hpx >= 2.f;
  vis = ok;
  cx = ok ? fmaf(0.25f * (pxs[0] + pxs[1] + pxs[2] + pxs[3]) - 0.5f, c.inv_half_res, -1.f) : 0.f;
  cy = ok ? fmaf(0.25f * (pys[0] + pys[1] + pys[2] + pys[3]) - 0.5f, c.inv_half_res, -1.f) : 0.f;
  area = ok ? fmaxf(0.5f * fabsf(a2) - 0.5f * per + 1.f, 0.f) * c.inv_res2 : 0.f;
  ratio = ok ? wpx * frcp(hpx) : 0.f;
}

// vision_mode = 1: the camera features as detect_rectangle (hover.py:157-222) reports them for the rendered frame, without
// rendering it.  The red box (front face panel[], back face panel_back[]) projects to a convex silhouette; for every pixel
// row the silhouette's x interval at the row's centre line is the min / max over the 12 box edges crossing it, which gives
// the covered columns [l, r].  From the row spans:
//   red_at_edges (hover.py:180-189)  a covered pixel in row / column 0 or res-1 rejects the frame
//   contourArea  (hover.py:206)      the contour runs through the centres of the border pixels (blob pixels with a
//                                    background 4-neighbour), so by Pick's theorem its area is N - B/2 - 1
//   boundingRect (hover.py:209-213)  covered columns x covered rows
//   centre       (hover.py:197-203)  mean of the projected front-face corners - 0.5 px (stand-in for the mean of the
//                                    approxPolyDP corners: within 0.8 px, tests/test_oracle_golden.py)
// oracle/vision.py:raster_features is the float64 statement of this function and equals the reference's detector on 1000
// rasterised frames (visibility, area, ratio exactly).  Not inlined: it runs once per agent step and only in this mode.
// (its constants live in a small device buffer: passing the DevConfig by reference would force the specialised kernels to
// materialise their literal-folded copy of it in local memory, and 35 by-value arguments would cost the callers registers)
struct RasterConsts { float cam_sd, cam_cd, inv_tan, res, half_res, inv_half_res, inv_res2, cam_near, cam_off[3], pad, panel[12], panel_back[12]; };

// The two steps of the silhouette raster that vision_raster and the camera-frame kernel share, so that a drawn frame covers
// exactly the pixels vision_raster counts.  raster_project: the 8 box corners (front face, then back face) in camera space --
// xr right, yu up, dep along the view axis -- and in continuous pixel coordinates (row 0 = top); returns whether every corner
// is in front of the near plane (otherwise pxs / pys of the corners behind it are meaningless).
QX_DI bool raster_project(const RasterConsts& c, const float px_w, const float py_w, const float pz_w, const float x, const float y,
                          const float z, const float w, float (&pxs)[8], float (&pys)[8], float (&xrs)[8], float (&yus)[8], float (&deps)[8]) {
  const float* panel_front = c.panel;
  const float* panel_back = c.panel_back;
  const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, xz = x * z, yz = y * z, wx = w * x, wy = w * y, wz = w * z;
  const float r00 = 1.f - 2.f * (yy + zz), r01 = 2.f * (xy - wz), r02 = 2.f * (xz + wy);
  const float r10 = 2.f * (xy + wz), r11 = 1.f - 2.f * (xx + zz), r12 = 2.f * (yz - wx);
  const float r20 = 2.f * (xz - wy), r21 = 2.f * (yz + wx), r22 = 1.f - 2.f * (xx + yy);
  float sph = 0.f, cph = 1.f;
  if (fabsf(r20) < 0.99999f) {
    const float inv = frsqrt(r21 * r21 + r22 * r22);
    sph = r21 * inv; cph = r22 * inv;
  }
  const float sd = c.cam_sd, cd = c.cam_cd;
  const float fx = cd, fy = sd * sph, fzz = sd * cph;
  const float ux = -sd * cph, uy = sph * cph * (cd - 1.f), uz = fmaf(sph, sph, cd * cph * cph);
  const float rx = fy * uz - fzz * uy, ry = fzz * ux - fx * uz, rz = fx * uy - fy * ux;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float* P = k < 4 ? &panel_front[3 * k] : &panel_back[3 * (k - 4)];
    const float dx = P[0] - px_w, dy = P[1] - py_w, dz = P[2] - pz_w;
    const float bx = r00 * dx + r10 * dy + r20 * dz - c.cam_off[0];
    const float by = r01 * dx + r11 * dy + r21 * dz - c.cam_off[1];
    const float bz = r02 * dx + r12 * dy + r22 * dz - c.cam_off[2];
    const float depth = fx * bx + fy * by + fzz * bz;
    ok = ok && (depth > c.cam_near);
    const float k1 = c.inv_tan / fmaxf(depth, 1e-9f);
    const float xr = rx * bx + ry * by + rz * bz;
    pxs[k] = fmaf(xr * k1, c.half_res, c.half_res);
    const float yu = ux * bx + uy * by + uz * bz;
    pys[k] = fmaf(-yu * k1, c.half_res, c.half_res);
    xrs[k] = xr; yus[k] = yu; deps[k] = depth;
  }
  return ok;
}

// the 12 box edges (front ring, back ring, connectors) of projected corners, set up for raster_row_span
struct RasterEdges { float ex0[12], ey0[12], ey1[12], esl[12]; };
QX_DI void raster_edges(const float (&pxs)[8], const float (&pys)[8], RasterEdges& E) {
  constexpr int ea[12] = {0, 1, 2, 3, 4, 5, 6, 7, 0, 1, 2, 3}, eb[12] = {1, 2, 3, 0, 5, 6, 7, 4, 4, 5, 6, 7};
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    E.ex0[k] = pxs[ea[k]]; E.ey0[k] = pys[ea[k]]; E.ey1[k] = pys[eb[k]];
    const float dy = E.ey1[k] - E.ey0[k];
    E.esl[k] = dy != 0.f ? (pxs[eb[k]] - pxs[ea[k]]) / dy : 0.f;
  }
}

// covered columns [ln, rn] of pixel row r (empty: ln > rn): the silhouette's x interval on the row's centre line y = r + 0.5 is
// the min / max over the edges crossing it, and a pixel is covered when its centre x + 0.5 lies in that interval
QX_DI void raster_row_span(const RasterEdges& E, const int r, int& ln, int& rn) {
  ln = 1; rn = 0;
  const float yl = (float)r + 0.5f;
  float xl = 3.0e38f, xr = -3.0e38f;
#pragma unroll
  for (int k = 0; k < 12; ++k) {
    if ((E.ey0[k] - yl) * (E.ey1[k] - yl) <= 0.f && E.ey0[k] != E.ey1[k]) {
      const float xi = fmaf(yl - E.ey0[k], E.esl[k], E.ex0[k]);
      xl = fminf(xl, xi); xr = fmaxf(xr, xi);
    }
  }
  if (xl <= xr) { ln = (int)ceilf(xl - 0.5f); rn = (int)floorf(xr - 0.5f); }
}

static __device__ __noinline__ void vision_raster(const float px_w, const float py_w, const float pz_w, const float x, const float y, const float z,
                                                  const float w, const float* __restrict__ consts, bool& vis, float& cx, float& cy, float& area, float& ratio) {
  const RasterConsts c = *reinterpret_cast<const RasterConsts*>(consts);
  float pxs[8], pys[8], xrs[8], yus[8], deps[8];
  const bool ok = raster_project(c, px_w, py_w, pz_w, x, y, z, w, pxs, pys, xrs, yus, deps);
  vis = false; cx = cy = area = ratio = 0.f;
  if (!ok) return;
  float ymin = pys[0], ymax = pys[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) { ymin = fminf(ymin, pys[k]); ymax = fmaxf(ymax, pys[k]); }
  const int res = (int)c.res;
  int r0 = (int)ceilf(ymin - 0.5f), r1 = (int)floorf(ymax - 0.5f);
  r0 = max(r0, -1); r1 = min(r1, res);  // rows outside the image only matter as "touches the border"
  RasterEdges E;
  raster_edges(pxs, pys, E);
  int n_pix = 0, interior = 0, lmin = 1 << 20, rmax = -(1 << 20), first = 1 << 20, last = -(1 << 20);
  int lp = 1, rp = 0, lc = 1, rc = 0;  // spans of the previous and the current row (empty: l > r)
  bool edge = false;
  for (int r = r0; r <= r1 + 1; ++r) {  // one row ahead: the interior count of a row needs its lower neighbour
    int ln = 1, rn = 0;
    if (r <= r1) {
      raster_row_span(E, r, ln, rn);
      if (ln <= rn) {
        n_pix += rn - ln + 1;
        lmin = min(lmin, ln); rmax = max(rmax, rn); first = min(first, r); last = max(last, r);
        edge = edge || r <= 0 || r >= res - 1 || ln <= 0 || rn >= res - 1;
      }
    }
    if (lc <= rc && lp <= rp && ln <= rn) interior += max(0, min(min(rc - 1, rp), rn) - max(max(lc + 1, lp), ln) + 1);
    lp = lc; rp = rc; lc = ln; rc = rn;
  }
  if (n_pix == 0 || edge) return;
  const int wpx = rmax - lmin + 1, hpx = last - first + 1;
  if (wpx < 2 || hpx < 2) return;
  vis = true;
  area = ((float)n_pix - 0.5f * (float)(n_pix - interior) - 1.f) * c.inv_res2;
  ratio = (float)wpx / (float)hpx;
  cx = fmaf(0.25f * (pxs[0] + pxs[1] + pxs[2] + pxs[3]) - 0.5f, c.inv_half_res, -1.f);
  cy = fmaf(0.25f * (pys[0] + pys[1] + pys[2] + pys[3]) - 0.5f, c.inv_half_res, -1.f);
}

// yaw task: centre of the red sphere (main.py:16-23, radius 0.1 at (2,0,1); yaw.py:63 detect_red_sphere_center is
// missing from the reference) projected through the same FPV camera model; (0,0) when it is not in the image.
__device__ __forceinline__ void vision_point(const Env& e, const DevConfig& c, bool& vis, float& cx, float& cy) {
  const float x = e.qx, y = e.qy, z = e.qz, w = e.qw;
  const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, xz = x * z, yz = y * z, wx = w * x, wy = w * y, wz = w * z;
  const float r00 = 1.f - 2.f * (yy + zz), r01 = 2.f * (xy - wz), r02 = 2.f * (xz + wy);
  const float r10 = 2.f * (xy + wz), r11 = 1.f - 2.f * (xx + zz), r12 = 2.f * (yz - wx);
  const float r20 = 2.f * (xz - wy), r21 = 2.f * (yz + wx), r22 = 1.f - 2.f * (xx + yy);
  float sph = 0.f, cph = 1.f;
  if (fabsf(r20) < 0.99999f) {
    const float inv = frsqrt(r21 * r21 + r22 * r22);
    sph = r21 * inv; cph = r22 * inv;
  }
  const float sd = c.cam_sd, cd = c.cam_cd;
  const float fx = cd, fy = sd * sph, fzz = sd * cph;
  const float ux = -sd * cph, uy = sph * cph * (cd - 1.f), uz = fmaf(sph, sph, cd * cph * cph);
  const float rx = fy * uz - fzz * uy, ry = fzz * ux - fx * uz, rz = fx * uy - fy * ux;
  const float dx = c.panel[0] - e.px, dy = c.panel[1] - e.py, dz = c.panel[2] - e.pz;
  const float bx = r00 * dx + r10 * dy + r20 * dz - c.cam_off[0];
  const float by = r01 * dx + r11 * dy + r21 * dz - c.cam_off[1];
  const float bz = r02 * dx + r12 * dy + r22 * dz - c.cam_off[2];
  const float depth = fx * bx + fy * by + fzz * bz;
  const float k1 = c.inv_tan * frcp(fmaxf(depth, 1e-9f));
  const float px = fmaf((rx * bx + ry * by + rz * bz) * k1, c.half_res, c.half_res);
  const float py = fmaf(-(ux * bx + uy * by + uz * bz) * k1, c.half_res, c.half_res);
  vis = depth > c.cam_near && px >= 0.f && px <= c.res && py >= 0.f && py <= c.res;
  cx = vis ? fmaf(px, c.inv_half_res, -1.f) : 0.f;
  cy = vis ? fmaf(py, c.inv_half_res, -1.f) : 0.f;
}

// Aviary(start_pos, start_orn) + Aviary.reset() + the env bookkeeping of
// hover.py:98-107.  prev_action is deliberately left alone (hover.py:31,357).
__device__ __forceinline__ void respawn(Env& e, const DevConfig& c, uint32_t k0, uint32_t k1) {
  float px = c.start_pos[0], py = c.start_pos[1], pz = c.start_pos[2], yaw = c.start_rpy[2];
  if (c.spawn_pos_noise != 0.f || c.spawn_yaw_noise != 0.f) {
    const uint4 b = env_philox(make_uint4(0u, STREAM_SPAWN, e.rng_ctr, 0u), k0, k1);
    px = fmaf(c.spawn_pos_noise, 2.f * u01(b.x) - 1.f, px);
    py = fmaf(c.spawn_pos_noise, 2.f * u01(b.y) - 1.f, py);
    pz = fmaf(c.spawn_pos_noise, 2.f * u01(b.z) - 1.f, pz);
    yaw = fmaf(c.spawn_yaw_noise, 2.f * u01(b.w) - 1.f, yaw);
  }
  pz = fmaxf(pz, c.floor_z);
  e.px = px; e.py = py; e.pz = pz;
  float sr, cr, sp, cp, sy, cy;
  sincosf(0.5f * c.start_rpy[0], &sr, &cr);
  sincosf(0.5f * c.start_rpy[1], &sp, &cp);
  sincosf(0.5f * yaw, &sy, &cy);
  e.qx = sr * cp * cy - cr * sp * sy;
  e.qy = cr * sp * cy + sr * cp * sy;
  e.qz = cr * cp * sy - sr * sp * cy;
  e.qw = cr * cp * cy + sr * sp * sy;
  e.vx = e.vy = e.vz = 0.f;
  e.wx = e.wy = e.wz = 0.f;
#pragma unroll
  for (int m = 0; m < 4; ++m) e.thr[m] = c.spawn_thr;
#pragma unroll
  for (int a = 0; a < 3; ++a) { e.pi[a] = 0.f; e.pe[a] = 0.f; e.swb[a] = 0.f; e.svb[a] = 0.f; }
  e.sqx = e.qx; e.sqy = e.qy; e.sqz = e.qz; e.sqw = e.qw; e.spx = px; e.spy = py; e.spz = pz;
  e.contact = pz <= c.floor_z;
  e.flags = 0u;
  e.step_count = 0;
  e.pcx = e.pcy = e.parea = e.pratio = 0.f;
  e.ep_ret = 0.f;
  if (c.task == 1) { e.pa[0] = e.pa[1] = e.pa[2] = e.pa[3] = 0.f; }  // yaw.py:90-92 clears the action history
}

}  // namespace qx
