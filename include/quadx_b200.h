/*
 * quadx_b200.h -- C-ABI of the B200-native batched QuadX hover / yaw simulator.
 *
 * This is the drop-in boundary for the reference's env step path
 * (SURVEY.md 8b).  Each entry point names the reference interface it replaces
 * (paths relative to the reference repository root).  The library is
 * libquadx_b200.so, built by fpv-drone-rl-agent_b200/csrc/build.py for sm_100a only.
 *
 * Conventions
 *   - every function returns 0 on success, a negative QX_E* code otherwise and
 *     never throws; qx_last_error() gives the text of the last failure of the
 *     calling thread.
 *   - pointers named *_dev are device pointers on the handle's device; work is
 *     enqueued on the cudaStream_t passed as `stream` (a void* here so the
 *     header needs no CUDA include) and is NOT synchronised.
 *   - pointers named *_host are ordinary host pointers; those calls copy
 *     through pinned staging buffers owned by the handle and return after the
 *     results are in host memory.
 *   - device buffers of qx_reset / qx_step / qx_step_begin / qx_step_end / qx_step_k are accessed with vector
 *     instructions and must be aligned accordingly, else the call returns QX_EINVAL and launches nothing:
 *     obs_dev 16-byte (QX_OBS_F32) / 8-byte (QX_OBS_BF16) aligned when obs_stride is a multiple of 4 (any
 *     other stride is written element by element, at any element-aligned address); hover actions_dev and
 *     terminal_obs_dev 16-byte aligned.  cudaMalloc'd buffers and whole torch tensors are; a column view
 *     such as buf[:, 1:21] of a [n, 24] f32 buffer is not.
 *   - a handle is not thread-safe; independent handles are.
 *   - one env == one drone in its own world (hover.py:78: one drone per Aviary).
 */
#ifndef QUADX_B200_H
#define QUADX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QX_VERSION 2
#define QX_OBS_DIM_HOVER 20 /* hover.py:67 */
#define QX_OBS_DIM_YAW 12   /* yaw.py:41-45 */
#define QX_ACT_DIM_HOVER 4  /* hover.py:59-61 */
#define QX_ACT_DIM_YAW 1    /* yaw.py:37 */
#define QX_STATE_WORDS 44   /* carried words per env (11 float4 planes) */
#define QX_STATE_WORDS_CASCADE 68 /* ... when flight_mode != 0: + 6 planes of outer-loop PID memory */

enum { QX_OK = 0, QX_EINVAL = -1, QX_ECUDA = -2, QX_ENOMEM = -3, QX_EARCH = -4 };
enum { QX_TASK_HOVER = 0, QX_TASK_YAW = 1 };
enum { QX_OBS_F32 = 0, QX_OBS_BF16 = 1 };
#define QX_FRAME_RGBA 0
#define QX_FRAME_MASK 1

/* Parameters of one simulation.  Defaults (qx_default_config) are the literals
 * of hover.py:23-51,77-110, cf2x.yaml:1-19 and cf2x.urdf:10-68; every field the
 * PyFlyt/pybullet restatement is unsure about is data here, not code. */
typedef struct QxConfig {
  int32_t task;               /* QX_TASK_*                                     */
  /* --- drone: cf2x.urdf / cf2x.yaml ---------------------------------------- */
  float mass;                 /* cf2x.urdf:10                                  */
  float inertia[3];           /* cf2x.urdf:12                                  */
  float motor_x[4];           /* cf2x.urdf:35,46,57,68                         */
  float motor_y[4];
  float torque_sign[4];       /* reaction torque sign per motor                */
  float motor_map[16];        /* row-major [motor][roll,pitch,yaw,thrust]      */
  float total_thrust;         /* cf2x.yaml:2                                   */
  float thrust_coef;          /* cf2x.yaml:3                                   */
  float torque_coef;          /* cf2x.yaml:4                                   */
  float noise_ratio;          /* cf2x.yaml:5                                   */
  float tau;                  /* cf2x.yaml:6                                   */
  float drag_coef_xyz;        /* cf2x.yaml:9                                   */
  float drag_area_xyz;        /* cf2x.yaml:10                                  */
  float drag_coef_pqr;        /* cf2x.yaml:11                                  */
  float air_density;
  float rate_kp[3];           /* cf2x.yaml:16                                  */
  float rate_ki[3];           /* cf2x.yaml:17                                  */
  float rate_kd[3];           /* cf2x.yaml:18                                  */
  float rate_lim[3];          /* cf2x.yaml:19                                  */
  float pwm_idle;
  float physics_hz;           /* hover.py:23                                   */
  float control_hz;           /* PyFlyt QuadX default                          */
  float gravity;
  int32_t state_stale;        /* Aviary.state is one sub-step stale            */
  int32_t gyro;               /* gyroscopic term                               */
  float max_coord_vel;        /* btMultiBody velocity clamp                    */
  float floor_z;              /* declared floor stand-in                       */
  /* --- camera + target: hover.py:84-87,116-155 ------------------------------ */
  float cam_tilt_up_deg;
  float cam_fov_deg;
  float cam_res;
  float cam_near;
  float cam_offset[3];
  float vis_margin_px;
  float panel[12];            /* 4 corners of the red face, world xyz          */
  /* --- env: hover.py:23-51 -------------------------------------------------- */
  int32_t aviary_steps_per_step; /* hover.py:24 env_step_ratio (yaw.py:126: 1) */
  int32_t max_steps;          /* hover.py:35                                   */
  int32_t floor_grace_steps;  /* hover.py:283                                  */
  int32_t reset_idle_steps;   /* hover.py:109                                  */
  float agent_dt;             /* hover.py:25                                   */
  float flight_dome_size;     /* hover.py:37                                   */
  float floor_threshold;      /* hover.py:38                                   */
  float target_area;          /* hover.py:50                                   */
  float target_ratio;         /* hover.py:51                                   */
  float action_scale[3];      /* hover.py:338-340                              */
  float start_pos[3];         /* hover.py:78                                   */
  float start_rpy[3];         /* hover.py:79                                   */
  float spawn_throttle;       /* addition: motors pre-spun (0 = reference)     */
  float spawn_pos_noise;      /* addition: Philox reset noise (0 = reference)  */
  float spawn_yaw_noise;      /* yaw.py:79 uses U(-pi, pi)                     */
  int32_t render;             /* hover.py:283: floor rule off when rendering   */
  int32_t auto_reset;         /* SB3 VecEnv semantics (train_hover.py:42)      */
  int32_t noise;              /* motor noise on/off                            */
  /* --- flight modes: hover.py:13,19 takes flight_mode and never uses it (set_mode(0) is literal at :92), so 0
   * is the reference's behaviour.  Non-zero selects the rest of PyFlyt's QuadX.set_mode cascade over the
   * gains of cf2x.yaml:21-53 (hover task only):  -1 motor pwm | 0 vp,vq,vr,T | 1 p,q,r,vz | 2 vp,vq,vr,z |
   * 3 p,q,r,z | 4 u,v,vr,z | 5 u,v,vr,vz | 6 vx,vy,vr,vz | 7 x,y,r,z.  setpoint = (action_scale * a[0..2],
   * thrust_scale * a[3] + thrust_bias); in mode -1 all four channels use the thrust mapping. ---------------- */
  int32_t flight_mode;
  float thrust_scale;         /* hover.py:341 (a3 + 1) / 2  ->  0.5                */
  float thrust_bias;          /*                               0.5                */
  float att_pid[12];          /* ang_pos kp[3] ki[3] kd[3] lim[3], cf2x.yaml:21-26 */
  float vel_pid[8];           /* lin_vel kp[2] ki[2] kd[2] lim[2], cf2x.yaml:28-33 */
  float pos_pid[8];           /* lin_pos kp[2] ki[2] kd[2] lim[2], cf2x.yaml:35-40 */
  float zpos_pid[4];          /* z_pos kp ki kd lim,               cf2x.yaml:42-47 */
  float zvel_pid[4];          /* z_vel kp ki kd lim,               cf2x.yaml:49-54 */
  /* --- camera features (hover.py:157-222).  0: analytic projection of the four front-face corners with pixel-lattice
   * corrections (default, cheapest).  1: scan conversion of the box silhouette on the 128 x 128 lattice and the contour
   * features as cv2 reports them for the rendered frame -- visibility, contour area and bounding-box ratio equal the
   * reference's detect_rectangle on rasterised frames; ~1.5x the step cost.  qx_render draws the frame in either mode (its
   * pixels are the ones mode 1 counts). ----------------------------------------------------------------------------------- */
  int32_t vision_mode;
  float panel_back[12];       /* the 4 corners of the box face behind panel[] (hover.py:118-147: 0.04 deep) */
} QxConfig;

typedef struct QxHandle QxHandle;

/* Fill *cfg with the reference's literals for `task`. */
int qx_default_config(int32_t task, QxConfig* cfg);

/* Replaces: QuadXHoverEnv.__init__ (hover.py:11-70) x n_envs and the 16-process
 * SubprocVecEnv of train_hover.py:41-42.  env_id0 is the global index of the
 * first env of this shard: the Philox key of env i is (seed, env_id0 + i), so
 * results do not depend on how envs are split over GPUs. */
int qx_create(const QxConfig* cfg, int64_t n_envs, uint64_t seed, uint64_t env_id0, int device, QxHandle** out);

/* Replaces: QuadXHoverEnv.close (hover.py:363-365). */
int qx_destroy(QxHandle* h);

/* Replaces: QuadXHoverEnv.reset (hover.py:72-114) for the envs whose mask byte
 * is non-zero (all when mask_dev is NULL).  obs_dev: [n_envs, obs_stride]
 * elements of obs_dtype, written only for the reset envs; may be NULL. */
int qx_reset(QxHandle* h, const uint8_t* mask_dev, void* obs_dev, int32_t obs_dtype, int64_t obs_stride, void* stream);

/* Replaces: QuadXHoverEnv.step (hover.py:334-358) for every env, plus the
 * VecEnv auto-reset when cfg.auto_reset: on done the obs written is the first
 * obs of the next episode and terminal_obs_dev (nullable, f32 [n, obs_dim])
 * receives the last obs of the finished one.
 *   actions_dev  f32 [n_envs, act_dim]
 *   obs_dev      obs_dtype [n_envs, obs_stride]
 *   reward_dev   f32 [n_envs]; terminated_dev / truncated_dev  u8 [n_envs] */
int qx_step(QxHandle* h, const float* actions_dev, void* obs_dev, int32_t obs_dtype, int64_t obs_stride,
            float* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev, void* stream);

/* qx_step in two halves, for callers that need the finished envs between the step and their reset (the PPO
 * rollout bootstraps truncated episodes from terminal_obs there): qx_step_begin runs the step and queues the
 * finished envs, qx_step_end re-creates them and writes their first observation.  qx_step == begin + end in effect;
 * for batches of <= 16 384 envs (latency-bound) qx_step does both in one launch instead of two.
 * qx_done_queue gives the device addresses of the queue (count, env indices) of the step just taken: valid from qx_step_begin
 * until the next step, also while qx_step_end runs -- a consumer of the queue may run concurrently with the reset on another stream. */
int qx_step_begin(QxHandle* h, const float* actions_dev, void* obs_dev, int32_t obs_dtype, int64_t obs_stride,
                  float* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev, float* terminal_obs_dev, void* stream);
int qx_step_end(QxHandle* h, void* obs_dev, int32_t obs_dtype, int64_t obs_stride, void* stream);
int qx_done_queue(QxHandle* h, const uint32_t** count_dev, const uint32_t** idx_dev);

/* The FPV camera frame (Camera.capture_image -> drones[0].rgbaImg, read by detect_rectangle hover.py:157-222) of m envs,
 * drawn from their current pose: frames_dev u8 [m, res, res, 4] (RGBA) or [m, res, res] (MASK), res = cfg.cam_res.
 * env_idx_dev: int32 [m] device indices, or NULL for all envs (m must then equal n_envs); an index outside [0, n_envs)
 * gets a background frame.  Hover task only.  Enqueued on `stream`, no synchronisation, graph-capturable.
 * frames_dev must be 16-byte aligned (the frames are written with 16-byte stores).  Row 0 is the top of the image.
 * RGBA: box (200, 0, 0, 255) on (170, 190, 230, 255); MASK: 255 on the box, 0 elsewhere (hover.py:173-177's red mask).  A pixel is on the box when its centre is inside the box's silhouette -- the pixels
 * vision_mode = 1 counts; a box crossing the camera's near plane is clipped to it. */
int qx_render(QxHandle* h, const int32_t* env_idx_dev, int64_t m, int32_t fmt, uint8_t* frames_dev, void* stream);

/* k consecutive qx_step in one launch with the state kept in registers
 * (physics-only benchmarking, SURVEY 8d): actions_dev f32 [k, n, act_dim],
 * obs_dev f32 [k, n, obs_dim], reward_dev [k, n], terminated/truncated [k, n]. */
int qx_step_k(QxHandle* h, int32_t k, const float* actions_dev, float* obs_dev, float* reward_dev,
              uint8_t* terminated_dev, uint8_t* truncated_dev, void* stream);

/* Host-buffer variants of reset / step: the call a reference-side binding makes
 * when it owns numpy arrays (copies H2D / D2H inside, returns synchronised). */
int qx_reset_host(QxHandle* h, const uint8_t* mask_host, float* obs_host);
int qx_step_host(QxHandle* h, const float* actions_host, float* obs_host, float* reward_host,
                 uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host);
/* qx_step_host with the observation element type chosen by the caller: QX_OBS_BF16 halves the bytes that cross PCIe
 * (the call is bound by the device-to-host copy: 80 of its 86 result bytes per env-step are the observation; a bf16
 * policy input loses nothing, tests/test_gpu_properties.py holds "bf16 obs == rounded f32 obs").  obs_host is
 * [n_envs, obs_dim] of that type; everything else as qx_step_host.  Pinned caller buffers are written in place. */
int qx_step_host_ex(QxHandle* h, const float* actions_host, void* obs_host, int32_t obs_dtype, float* reward_host,
                    uint8_t* terminated_host, uint8_t* truncated_host, float* terminal_obs_host);

/* Carried state as qx_state_words(h) planes of n_envs 32-bit words (layout in
 * DESIGN.md; QX_STATE_WORDS, or QX_STATE_WORDS_CASCADE when cfg.flight_mode != 0);
 * for parity tests and checkpoint/resume. */
int qx_get_state(QxHandle* h, void* planes_host);
int qx_set_state(QxHandle* h, const void* planes_host);
/* The flags word of envs [first, first + count) (bit 0 contact, 1 terminated, 2 truncated, 3 out_of_bounds, 4 on_floor,
 * 5 low-z): what the `info` dict of hover.py:53-57,280,289 is made of.  Synchronous, one word per env. */
int qx_get_flags(QxHandle* h, int64_t first, int64_t count, uint32_t* flags_host);
int32_t qx_state_words(const QxHandle* h);

/* Replaces: SB3 Monitor's info["episode"] (train_hover.py:42 make_vec_env):
 * sums over the episodes finished since the last call with clear != 0. */
int qx_episode_stats(QxHandle* h, double* sum_return, int64_t* sum_length, int64_t* n_episodes, int32_t clear);

/* Evaluation ledger (SB3 evaluate_policy / Monitor per episode; test_hover.py:13-27): for a handle created with
 * cfg.auto_reset == 0, call after every qx_step.  Env i whose record is open (end_dev[i] == 0) and whose episode has
 * ended (flags word: terminated | truncated) closes it: ret_dev[i] = its episode return (the ep_ret word), len_dev[i] =
 * step_count, end_dev[i] = the flags word (bits as qx_get_flags; never 0 once closed), and *n_closed_dev += 1.
 * Closed records are never written again.  The caller zero-fills end_dev and *n_closed_dev before the first step.
 * ret_dev f32 [n_envs], len_dev i32 [n_envs], end_dev u32 [n_envs], n_closed_dev u32 [1].  Any task, flight or vision
 * mode.  Enqueued on `stream`, no allocation, no synchronisation, graph-capturable; QX_EINVAL (nothing launched) for a
 * null handle, a handle with auto_reset != 0 or a null output. */
int qx_episode_record(QxHandle* h, float* ret_dev, int32_t* len_dev, uint32_t* end_dev, uint32_t* n_closed_dev, void* stream);

/* Failure detection (no reference counterpart): envs whose state stopped being finite since creation; each was
 * terminated like an out-of-bounds flight and re-created by the auto-reset. */
int qx_nonfinite_count(QxHandle* h, int64_t* count);

int64_t qx_num_envs(const QxHandle* h);
int32_t qx_obs_dim(const QxHandle* h);
int32_t qx_act_dim(const QxHandle* h);
/* device pointer to the qx_state_words(h) / 4 float4 state planes (plane stride = n_envs) */
void* qx_state_ptr(QxHandle* h);
/* 1 when the handle runs the kernels specialised for the reference's own parameter set (the model constants of
 * qx_default_config(QX_TASK_HOVER) compiled in as literals); any other configuration -- or QX_FORCE_GENERIC=1 in the
 * environment at qx_create -- runs the generic kernels that read every constant from the config.  Same results. */
int32_t qx_uses_reference_constants(const QxHandle* h);
int32_t qx_config_matches_reference_constants(const QxConfig* cfg);
/* number of kernels this library has launched in the calling process */
int64_t qx_launch_count(void);
/* sizeof(QxConfig) as compiled into the library (binding self-check) */
int64_t qx_sizeof_config(void);
const char* qx_last_error(void);
int32_t qx_version(void);

/* Environment variables read once at qx_create (tuning and A/B measurements; every setting computes the same results, and the
 * defaults are what measured fastest on B200 -- profiles/k1_r2_variants.md):
 *   QX_FORCE_GENERIC=1   generic kernels even when the configuration equals the reference's constants
 *   QX_HOT=0|1           never / always the lean one-step hover kernel (default: batches of >= 32 768 envs)
 *   QX_LANES=1|2|4       hot kernel: scalar lanes / two envs per thread on f32x2 / one env per thread, own components paired (default 4)
 *   QX_SHAPE=0|3|4|5     hot kernel launch shape (resident blocks per SM; default 4 = 5 blocks of 128 threads, 96 registers)
 *   QX_MERGED=1          hot kernel also drains the reset queue (one launch per step; default 0: two launches)
 *   QX_PAIRED_RESET=0    queued envs re-created by the generic code instead of the paired one
 *   QX_STREAM_STORES=1|2 evict-first stores for the outputs / the state planes too (default 0)
 *   QX_PDL=0             no programmatic dependent launches (default 1: the reset-queue kernel of qx_step, and consecutive
 *                        single-launch steps, are scheduled while their predecessor still runs and wait for it on the device)
 *   QX_HOST_CHUNKS=k     *_host calls: k equal pieces (the first halved again), k < 0: -k geometric pieces (default: 5 geometric)
 *   QX_HOST_ONE_D2H=1    *_host calls: the small result arrays share the observation's device-to-host stream */

#ifdef __cplusplus
}
#endif
#endif /* QUADX_B200_H */
