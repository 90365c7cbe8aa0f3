"""ctypes binding of libquadx_b200.so (include/quadx_b200.h).

There is no CPU fallback: if the library is missing or does not load, importing
the env classes raises.  The binding is deliberately thin -- torch is used only
for device memory, streams and torch.distributed."""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QX_LIB") or os.path.join(_HERE, "csrc", "libquadx_b200.so")  # QX_LIB: a tuning build (tools/ only)

QX_TASK_HOVER, QX_TASK_YAW = 0, 1
QX_OBS_F32, QX_OBS_BF16 = 0, 1
QX_FRAME_RGBA, QX_FRAME_MASK = 0, 1
QX_STATE_WORDS = 44
QX_STATE_WORDS_CASCADE = 68

f32, i32 = C.c_float, C.c_int32


class QxConfig(C.Structure):
    """Mirror of ``struct QxConfig`` in include/quadx_b200.h (field order matters)."""

    _fields_ = [
        ("task", i32),
        ("mass", f32), ("inertia", f32 * 3), ("motor_x", f32 * 4), ("motor_y", f32 * 4), ("torque_sign", f32 * 4),
        ("motor_map", f32 * 16), ("total_thrust", f32), ("thrust_coef", f32), ("torque_coef", f32), ("noise_ratio", f32),
        ("tau", f32), ("drag_coef_xyz", f32), ("drag_area_xyz", f32), ("drag_coef_pqr", f32), ("air_density", f32),
        ("rate_kp", f32 * 3), ("rate_ki", f32 * 3), ("rate_kd", f32 * 3), ("rate_lim", f32 * 3), ("pwm_idle", f32),
        ("physics_hz", f32), ("control_hz", f32), ("gravity", f32), ("state_stale", i32), ("gyro", i32),
        ("max_coord_vel", f32), ("floor_z", f32),
        ("cam_tilt_up_deg", f32), ("cam_fov_deg", f32), ("cam_res", f32), ("cam_near", f32), ("cam_offset", f32 * 3),
        ("vis_margin_px", f32), ("panel", f32 * 12),
        ("aviary_steps_per_step", i32), ("max_steps", i32), ("floor_grace_steps", i32), ("reset_idle_steps", i32),
        ("agent_dt", f32), ("flight_dome_size", f32), ("floor_threshold", f32), ("target_area", f32), ("target_ratio", f32),
        ("action_scale", f32 * 3), ("start_pos", f32 * 3), ("start_rpy", f32 * 3), ("spawn_throttle", f32),
        ("spawn_pos_noise", f32), ("spawn_yaw_noise", f32), ("render", i32), ("auto_reset", i32), ("noise", i32),
        ("flight_mode", i32), ("thrust_scale", f32), ("thrust_bias", f32), ("att_pid", f32 * 12), ("vel_pid", f32 * 8),
        ("pos_pid", f32 * 8), ("zpos_pid", f32 * 4), ("zvel_pid", f32 * 4),
        ("vision_mode", i32), ("panel_back", f32 * 12),
    ]

    def update(self, **kw) -> "QxConfig":
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError(f"QxConfig has no field {k!r}")
            cur = getattr(self, k)
            if isinstance(cur, C.Array):
                v = list(v)
                if len(v) != len(cur):
                    raise ValueError(f"{k}: expected {len(cur)} values")
                for i, x in enumerate(v):
                    cur[i] = x
            else:
                setattr(self, k, v)
        return self


class PpoPolicy(C.Structure):
    """Mirror of ``struct PpoPolicy`` in include/ppo_b200.h."""

    _fields_ = [("w1", C.c_void_p), ("w2p", C.c_void_p), ("w2v", C.c_void_p), ("w3", C.c_void_p), ("b1", C.c_void_p),
                ("b2", C.c_void_p), ("b3", C.c_void_p), ("log_std", C.c_void_p), ("obs_dim", i32), ("act_dim", i32)]


_lib = None


def lib() -> C.CDLL:
    """Load the CUDA library once; fail loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python fpv-drone-rl-agent_b200/csrc/build.py` "
            "(or __graft_entry__.build()). There is no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    vp, i64, u64, u8p, f32p = C.c_void_p, C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p
    protos = {
        "qx_default_config": (C.c_int, [i32, C.POINTER(QxConfig)]),
        "qx_create": (C.c_int, [C.POINTER(QxConfig), i64, u64, u64, C.c_int, C.POINTER(vp)]),
        "qx_destroy": (C.c_int, [vp]),
        "qx_reset": (C.c_int, [vp, u8p, vp, i32, i64, vp]),
        "qx_step": (C.c_int, [vp, f32p, vp, i32, i64, f32p, u8p, u8p, f32p, vp]),
        "qx_step_begin": (C.c_int, [vp, f32p, vp, i32, i64, f32p, u8p, u8p, f32p, vp]),
        "qx_step_end": (C.c_int, [vp, vp, i32, i64, vp]),
        "qx_done_queue": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
        "qx_step_k": (C.c_int, [vp, i32, f32p, f32p, f32p, u8p, u8p, vp]),
        "qx_render": (C.c_int, [vp, vp, i64, i32, u8p, vp]),
        "qx_reset_host": (C.c_int, [vp, u8p, f32p]),
        "qx_step_host": (C.c_int, [vp, f32p, f32p, f32p, u8p, u8p, f32p]),
        "qx_step_host_ex": (C.c_int, [vp, f32p, vp, i32, f32p, u8p, u8p, f32p]),
        "qx_get_state": (C.c_int, [vp, vp]),
        "qx_set_state": (C.c_int, [vp, vp]),
        "qx_get_flags": (C.c_int, [vp, i64, i64, vp]),
        "qx_episode_stats": (C.c_int, [vp, C.POINTER(C.c_double), C.POINTER(i64), C.POINTER(i64), i32]),
        "qx_episode_record": (C.c_int, [vp, f32p, vp, vp, vp, vp]),
        "qx_nonfinite_count": (C.c_int, [vp, C.POINTER(i64)]),
        "qx_num_envs": (i64, [vp]),
        "qx_obs_dim": (i32, [vp]),
        "qx_act_dim": (i32, [vp]),
        "qx_state_ptr": (vp, [vp]),
        "qx_state_words": (i32, [vp]),
        "qx_uses_reference_constants": (i32, [vp]),
        "qx_config_matches_reference_constants": (i32, [C.POINTER(QxConfig)]),
        "qx_launch_count": (i64, []),
        "qx_sizeof_config": (i64, []),
        "qx_last_error": (C.c_char_p, []),
        "qx_version": (i32, []),
        # include/ppo_b200.h
        "ppo_policy_forward": (C.c_int, [C.POINTER(PpoPolicy), vp, i64, i64, vp, vp, f32, u64, u64, u64, vp, i32, vp, vp, vp, vp, vp, vp]),
        "ppo_policy_forward_stats": (C.c_int, [C.POINTER(PpoPolicy), vp, i64, i64, vp, f32, vp, vp, vp, f32, u64, u64, u64, vp, i32, vp, vp, vp, vp, vp, i32, vp]),
        "ppo_bootstrap_truncated": (C.c_int, [C.POINTER(PpoPolicy), vp, i64, i64, vp, vp, f32, vp, vp, vp, vp, f32, vp, vp]),
        "ppo_bootstrap_truncated_first": (C.c_int, [C.POINTER(PpoPolicy), vp, i64, i64, vp, vp, f32, vp, vp, vp, vp, f32, vp, vp]),
        "ppo_gae": (C.c_int, [vp, vp, vp, vp, i32, i64, f32, f32, vp, vp, vp]),
        "ppo_running_stats_update": (C.c_int, [vp, i64, i64, i32, vp, f32, vp, vp, vp, vp]),
        "ppo_running_stats_scratch_bytes": (i64, [i32]),
        "ppo_reward_normalize": (C.c_int, [vp, vp, vp, vp, i64, f32, f32, f32, vp, vp, vp, vp, vp]),
        "ppo_reward_normalize_add": (C.c_int, [vp, vp, vp, vp, i64, f32, f32, f32, vp, vp, vp, vp, vp]),
        "ppo_test_gemm": (C.c_int, [vp, vp, vp, i32, i32, vp]),
        "ppo_test_gemm_mn": (C.c_int, [vp, vp, vp, i32, i32, i32, i32, vp]),
        "ppo_test_tanh_bf16": (C.c_int, [vp, vp, i64, vp]),
        "ppo_update_num_params": (i32, [i32, i32]),
        "ppo_update_workspace_bytes": (i64, [i32, i32]),
        "ppo_update_minibatch": (C.c_int, [C.POINTER(PpoPolicy), vp, vp, vp, vp, vp, vp, i32, i64, f32, f32, f32, i32, vp, vp, vp, vp]),
        "ppo_update_grad_norm": (C.c_int, [vp, i32, f32, vp, vp]),
        "ppo_update_adam": (C.c_int, [vp, vp, vp, vp, i32, f32, f32, f32, f32, f32, f32, C.POINTER(PpoPolicy), vp, vp]),
        "ppo_update_step_count": (C.c_int, [vp, i64, C.POINTER(i64), vp]),
        "ppo_update_set_lr_scale": (C.c_int, [vp, C.c_float, vp]),
        "ppo_update_recompute_logp": (C.c_int, [C.POINTER(PpoPolicy), vp, vp, vp, i32, i64, vp, vp, vp]),
        "ppo_update_kl_stop": (C.c_int, [vp, C.c_float, C.POINTER(i32), C.POINTER(i32), vp]),
        "ppo_update_set_log_std_floor": (C.c_int, [vp, i32, C.c_float, vp]),
        "qx_debug_clock_probe": (C.c_int, [vp, vp]),
    }
    for name, (res, args) in protos.items():
        fn = getattr(L, name)  # AttributeError here = header and library disagree
        fn.restype, fn.argtypes = res, args
    if L.qx_sizeof_config() != C.sizeof(QxConfig):
        raise ImportError(f"QxConfig layout mismatch: library {L.qx_sizeof_config()} B, binding {C.sizeof(QxConfig)} B")
    _lib = L
    return L


EXPORTED = [
    "qx_default_config", "qx_create", "qx_destroy", "qx_reset", "qx_step", "qx_step_begin", "qx_step_end", "qx_done_queue", "qx_step_k", "qx_render", "qx_reset_host", "qx_step_host", "qx_step_host_ex",
    "qx_get_state", "qx_set_state", "qx_get_flags", "qx_episode_stats", "qx_episode_record", "qx_nonfinite_count", "qx_num_envs", "qx_obs_dim", "qx_act_dim", "qx_state_ptr", "qx_state_words", "qx_uses_reference_constants", "qx_config_matches_reference_constants",
    "qx_launch_count", "qx_sizeof_config", "qx_last_error", "qx_version",
]
PPO_EXPORTED = ["ppo_policy_forward", "ppo_policy_forward_stats", "ppo_bootstrap_truncated", "ppo_bootstrap_truncated_first", "ppo_reward_normalize_add", "ppo_gae", "ppo_running_stats_update", "ppo_running_stats_scratch_bytes",
                "ppo_reward_normalize", "ppo_test_gemm", "ppo_test_gemm_mn", "ppo_test_tanh_bf16", "ppo_update_num_params", "ppo_update_workspace_bytes",
                "ppo_update_minibatch", "ppo_update_grad_norm", "ppo_update_adam", "ppo_update_step_count", "ppo_update_set_lr_scale", "ppo_update_kl_stop", "ppo_update_set_log_std_floor", "ppo_update_recompute_logp"]


class QxError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        raise QxError(f"libquadx_b200 error {rc}: {lib().qx_last_error().decode()}")


def default_config(task: int = QX_TASK_HOVER) -> QxConfig:
    cfg = QxConfig()
    check(lib().qx_default_config(task, C.byref(cfg)))
    return cfg


def ptr(t: torch.Tensor | None) -> C.c_void_p | None:
    return None if t is None else C.c_void_p(t.data_ptr())


def stream(device: torch.device) -> C.c_void_p:
    """The current stream of an indexed CUDA device (cuda_device), read as the raw handle (as torch's own generated launchers read
    it): building a torch.cuda.Stream object first costs a microsecond of host time on every eager launch."""
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(device.index))


def cuda_device(device: int | str | torch.device | None = None) -> torch.device:
    """None, "cuda", an int or a torch.device -> that CUDA device with its index, as tensors allocated there report it."""
    dev = torch.device("cuda") if device is None else torch.device(device)
    if dev.type != "cuda":
        raise ValueError(f"device must be a CUDA device, got {dev}")
    return dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())


def expect(t: torch.Tensor, name: str, *, dtype: torch.dtype | tuple, device: torch.device, shape=None, numel: int | None = None) -> None:
    """Raise ValueError naming `name` unless `t` is a contiguous tensor of `dtype` (or of one in a tuple) on `device`, with `shape`
    and `numel` where given: the kernels address such buffers densely from the base pointer and would misuse any other."""
    if ((t.dtype not in dtype if isinstance(dtype, tuple) else t.dtype != dtype) or t.device != device or not t.is_contiguous()
            or (shape is not None and tuple(t.shape) != tuple(shape)) or (numel is not None and t.numel() != numel)):
        raise ValueError(f"{name}: expected a contiguous tensor of {dtype}, shape {shape}, {numel} elements on {device}; got "
                         f"{t.dtype} {tuple(t.shape)} on {t.device} (contiguous: {t.is_contiguous()})")
