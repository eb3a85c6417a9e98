"""ctypes binding of libmrf_b200.so (include/mrf_b200.h).

There is no CPU fallback: if the CUDA library is missing, or no B200 is visible when a handle is created,
the call fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MRF_B200_LIB", os.path.join(_HERE, "libmrf_b200.so"))   # override: A/B builds only

MAX_ROBOTS, DOF, NLINKS, REC, OBST = 4, 7, 8, 44, 10
Q, QD, G0, W0, G1, W1, G2, W2, ANG, CON, RB = 0, 7, 14, 17, 18, 21, 22, 23, 24, 33, 37


class MrfError(RuntimeError):
    pass


class MrfConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("n_robots", C.c_int32), ("mode", C.c_int32), ("static_or_dyn", C.c_int32),
        ("has_collision_links", C.c_int32), ("estimate_goal", C.c_int32), ("estimate_robot", C.c_int32),
        ("reserved0", C.c_int32),
        ("estimate_horizon", C.c_double), ("dt", C.c_double), ("eps", C.c_double), ("jdot_sign", C.c_double),
        ("jdot_ref_sign", C.c_double), ("exec_scale", C.c_double),
        ("mount", (C.c_double * 16) * MAX_ROBOTS),
        ("limits", (C.c_double * 2) * DOF),
        ("r_robots", (C.c_double * NLINKS) * MAX_ROBOTS),
        ("dl_avg_vel_constant", C.c_double), ("dl_dist_constant", C.c_double),
        ("dl_goal_weight_follower", C.c_double), ("dl_goal_weight_leader", C.c_double),
        ("dl_nr_goal_scale", C.c_double), ("dl_dist_endeff", C.c_double), ("dl_backoff", C.c_double),
        ("dl_time_wait", C.c_int32), ("dl_time_gate", C.c_int32),
        ("collision_link_mask", C.c_int32 * MAX_ROBOTS),
    ]


class MrfEpisode(C.Structure):
    """include/mrf_b200.h: state of mrf_episode_step_dev_* (device pointers as integers)."""
    _fields_ = [
        ("struct_size", C.c_int32), ("n_horizon", C.c_int32), ("rollout_fabrics", C.c_int32),
        ("resolve_deadlocks", C.c_int32), ("n_per_link", C.c_int32), ("rollout_model", C.c_int32),
        ("epsilon", C.c_double), ("w1_rollout", C.c_double), ("w1_action", C.c_double),
        ("clearance_radius_sum", C.c_double), ("vel_limit", C.c_double * DOF),
        ("offsets", C.c_void_p), ("rec", C.c_void_p), ("goal0", C.c_void_p), ("w0", C.c_void_p), ("avg_vel", C.c_void_p),
        ("x_ee", C.c_void_p), ("goal_est", C.c_void_p), ("obst", C.c_void_p), ("spheres_x", C.c_void_p),
        ("action", C.c_void_p), ("kin_scratch", C.c_void_p), ("sm_state", C.c_void_p), ("time_step", C.c_void_p),
        ("time_deadlock_out", C.c_void_p), ("st_int", C.c_void_p), ("st_goal", C.c_void_p), ("flag", C.c_void_p),
        ("done_at", C.c_void_p), ("deadlock_steps", C.c_void_p), ("min_clearance", C.c_void_p),
        ("pick_and_place", C.c_int32), ("n_blocks", C.c_int32), ("blocks", C.c_void_p), ("start_goal", C.c_void_p),
        ("q_grip", C.c_void_p), ("goal_block", C.c_void_p), ("fsm_above", C.c_void_p), ("fsm_st", C.c_void_p),
        ("grip_action", C.c_void_p), ("nonfinite_steps", C.c_void_p),
    ]


class MrfPointEpisode(C.Structure):
    """include/mrf_b200.h: state of mrf_point_episode_run_dev_* (device pointers as integers)."""
    _fields_ = [
        ("struct_size", C.c_int32), ("n_robots", C.c_int32), ("dynamic", C.c_int32), ("n_scene", C.c_int32),
        ("epsilon", C.c_double), ("state", C.c_void_p), ("goal", C.c_void_p), ("weight", C.c_void_p),
        ("radius", C.c_void_p), ("scene", C.c_void_p), ("time_step", C.c_void_p), ("done_at", C.c_void_p),
        ("nonfinite_steps", C.c_void_p), ("min_clear_robots", C.c_void_p), ("min_clear_scene", C.c_void_p),
        ("traj", C.c_void_p),
    ]


_lib = None
_F = {"f32": (C.c_float, np.float32), "f64": (C.c_double, np.float64)}

# every symbol include/mrf_b200.h declares
EXPORTS = [
    "mrf_version", "mrf_last_error", "mrf_config_default", "mrf_create", "mrf_destroy", "mrf_device_count",
    "mrf_action_dev_f64", "mrf_action_dev_f32", "mrf_rollout_dev_f64", "mrf_rollout_dev_f32",
    "mrf_rollout_cart_dev_f64", "mrf_rollout_cart_dev_f32", "mrf_rollout_cart_all_dev_f64", "mrf_rollout_cart_all_dev_f32",
    "mrf_kinematics_dev_f64", "mrf_kinematics_dev_f32",
    "mrf_deadlock_dev_f64", "mrf_deadlock_dev_f32", "mrf_deadlock_rec_dev_f64", "mrf_deadlock_rec_dev_f32", "mrf_fsm_dev_f64", "mrf_fsm_dev_f32", "mrf_obstacles_dev_f64", "mrf_obstacles_dev_f32", "mrf_point_action_dev_f64", "mrf_point_action_dev_f32",
    "mrf_point_action_host_f64", "mrf_action_host_f64", "mrf_action_host_f32",
    "mrf_rollout_host_f64", "mrf_rollout_host_f32", "mrf_rollout_cart_host_f64", "mrf_rollout_cart_host_f32",
    "mrf_kinematics_host_f64", "mrf_deadlock_host_f64", "mrf_launch_count", "mrf_last_kernel_ms", "mrf_fma_peak", "mrf_set_coop_max_batch",
    "mrf_episode_step_dev_f64", "mrf_episode_step_dev_f32",
    "mrf_rollout_host_submit_f64", "mrf_rollout_host_submit_f32", "mrf_rollout_host_wait",
    "mrf_rollout_host_submit_compact_f64", "mrf_rollout_host_submit_compact_f32",
    "mrf_rfcv_post_dev_f32", "mrf_rfcv_post_dev_f64", "mrf_rollout_risk_dev_f32", "mrf_rollout_risk_dev_f64",
    "mrf_set_guard", "mrf_guard_stats", "mrf_rollout_static_dev_f32", "mrf_rollout_static_dev_f64",
    "mrf_rfcv_host_submit_f32", "mrf_point_episode_run_dev_f64", "mrf_point_episode_run_dev_f32",
]


def lib():
    """Load libmrf_b200.so (built by __graft_entry__.build()).  Raises MrfError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MrfError(f"{LIB_PATH} not found: build the CUDA library first (python -c 'import __graft_entry__ as g; "
                       "g.build()'); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.mrf_version.restype = C.c_int
    L.mrf_last_error.restype = C.c_char_p
    L.mrf_config_default.argtypes = [C.POINTER(MrfConfig), i32]
    L.mrf_create.argtypes = [C.POINTER(MrfConfig), i32, C.POINTER(vp)]
    L.mrf_destroy.argtypes = [vp]
    L.mrf_launch_count.argtypes = [vp]
    L.mrf_launch_count.restype = i64
    L.mrf_last_kernel_ms.argtypes = [vp]
    L.mrf_last_kernel_ms.restype = C.c_double
    for p in ("f32", "f64"):
        getattr(L, f"mrf_action_dev_{p}").argtypes = [vp, i32, i32, vp, i32, vp, vp, i64, vp]
        getattr(L, f"mrf_rollout_dev_{p}").argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_rollout_cart_dev_{p}").argtypes = [vp, i32, vp, i32, vp, i32, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_rollout_cart_all_dev_{p}").argtypes = [vp, vp, i32, vp, i32, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_kinematics_dev_{p}").argtypes = [vp, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_deadlock_dev_{p}").argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_deadlock_rec_dev_{p}").argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_fsm_dev_{p}").argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_obstacles_dev_{p}").argtypes = [vp, i32, vp, i32, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_action_host_{p}").argtypes = [vp, i32, i32, vp, i32, vp, vp, i64]
        getattr(L, f"mrf_rollout_host_{p}").argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, i64]
        getattr(L, f"mrf_rollout_cart_host_{p}").argtypes = [vp, i32, vp, i32, vp, i32, vp, vp, vp, i64]
        getattr(L, f"mrf_rfcv_post_dev_{p}").argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, i32]
        getattr(L, f"mrf_rollout_static_dev_{p}").argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, vp, vp, i64, vp]
        getattr(L, f"mrf_rollout_risk_dev_{p}").argtypes = [vp, vp, i32, vp, vp, vp, vp, i64, vp]
    L.mrf_rfcv_host_submit_f32.argtypes = [vp, vp, vp, i32, i32, vp, vp, i64]
    L.mrf_set_guard.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double, i64]
    L.mrf_guard_stats.argtypes = [vp, C.POINTER(C.c_int64)]
    L.mrf_point_action_dev_f64.argtypes = [vp, vp, i32, vp, i32, vp, vp, i64, vp]
    L.mrf_point_action_dev_f32.argtypes = [vp, vp, i32, vp, i32, vp, vp, i64, vp]
    L.mrf_point_action_host_f64.argtypes = [vp, vp, i32, vp, i32, vp, vp, i64]
    L.mrf_kinematics_host_f64.argtypes = [vp, vp, vp, vp, vp, vp, i64]
    L.mrf_deadlock_host_f64.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64]
    L.mrf_set_coop_max_batch.argtypes = [vp, i64]
    L.mrf_rollout_host_submit_f64.argtypes = [vp, vp, i32, vp, vp, vp, i64]
    L.mrf_rollout_host_submit_f32.argtypes = [vp, vp, i32, vp, vp, vp, i64]
    L.mrf_rollout_host_wait.argtypes = [vp, i32]
    L.mrf_rollout_host_submit_compact_f64.argtypes = [vp, vp, vp, i32, vp, vp, vp, i64]
    L.mrf_rollout_host_submit_compact_f32.argtypes = [vp, vp, vp, i32, vp, vp, vp, i64]
    L.mrf_episode_step_dev_f64.argtypes = [vp, C.POINTER(MrfEpisode), i64, vp]
    L.mrf_episode_step_dev_f32.argtypes = [vp, C.POINTER(MrfEpisode), i64, vp]
    L.mrf_point_episode_run_dev_f64.argtypes = [vp, C.POINTER(MrfPointEpisode), i64, i32, vp]
    L.mrf_point_episode_run_dev_f32.argtypes = [vp, C.POINTER(MrfPointEpisode), i64, i32, vp]
    L.mrf_fma_peak.argtypes = [vp, i32, C.POINTER(C.c_double)]
    _lib = L
    return L


def check(rc: int, what: str = "mrf"):
    if rc != 0:
        raise MrfError(f"{what} failed ({rc}): {lib().mrf_last_error().decode()}")


def default_config(n_robots: int, **overrides) -> MrfConfig:
    cfg = MrfConfig()
    check(lib().mrf_config_default(C.byref(cfg), n_robots), "mrf_config_default")
    for k, v in overrides.items():
        if k == "mount":
            for r, T in enumerate(v):
                flat = np.asarray(T, dtype=np.float64).reshape(16)
                for i in range(16):
                    cfg.mount[r][i] = flat[i]
        elif k == "limits":
            for i, (lo, hi) in enumerate(v):
                cfg.limits[i][0], cfg.limits[i][1] = lo, hi
        elif k == "collision_links":          # per robot a list of link numbers 1..8 (collision_links_nrs)
            for r, links in enumerate(v):
                cfg.collision_link_mask[r] = sum(1 << (int(l) - 1) for l in set(links))
        elif k == "r_robots":
            for r, row in enumerate(v):
                for l, x in enumerate(row):
                    cfg.r_robots[r][l] = float(x)
        else:
            if not hasattr(cfg, k):
                raise MrfError(f"unknown MrfConfig field {k}")
            setattr(cfg, k, v)
    return cfg


def hptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    return None if a is None else C.c_void_p(a.ctypes.data)


class Handle:
    """Owns one mrf_handle_t (one device).  Fails loudly if no B200 is visible."""

    def __init__(self, cfg: MrfConfig, device: int = 0):
        self.cfg = cfg
        self._h = C.c_void_p()
        check(lib().mrf_create(C.byref(cfg), device, C.byref(self._h)), "mrf_create")

    @property
    def ptr(self):
        return self._h

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().mrf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self) -> int:
        return int(lib().mrf_launch_count(self._h))

    def set_coop_max_batch(self, max_batch: int) -> None:
        """Batches up to max_batch use the cooperative low-latency rollout kernel (0 = never)."""
        check(lib().mrf_set_coop_max_batch(self._h, int(max_batch)), "mrf_set_coop_max_batch")

    def fma_peak_tflops(self, f64: bool = False) -> float:
        out = C.c_double(0.0)
        check(lib().mrf_fma_peak(self._h, int(f64), C.byref(out)), "mrf_fma_peak")
        return float(out.value)

    @property
    def last_kernel_ms(self) -> float:
        return float(lib().mrf_last_kernel_ms(self._h))
