"""Batched entry points over the C-ABI: numpy (host buffers) and torch (device tensors, hand-off only).

`Fabrics` owns one handle on one GPU.  Host methods take the reference's natural array-of-records order;
device methods take structure-of-arrays torch tensors (scenario index fastest) and launch on torch's current
stream.  Nothing here computes: every number comes out of libmrf_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import DOF, NLINKS, OBST, REC, Handle, MrfError, check, default_config, hptr, lib

_NP = {"f64": np.float64, "f32": np.float32}


def _arr(a, dtype, shape=None):
    a = np.ascontiguousarray(a, dtype=dtype)
    if shape is not None and tuple(a.shape) != tuple(shape):
        raise MrfError(f"expected array of shape {tuple(shape)}, got {tuple(a.shape)}")
    return a


def _chk(name, t, shape, dtype=None, device=None, optional=True):
    """Every tensor handed to the C-ABI as a raw pointer: right shape, dtype, device, contiguous -- otherwise the kernels
    would read or write out of bounds without any error."""
    if t is None:
        if optional:
            return None
        raise MrfError(f"{name} is required")
    if tuple(t.shape) != tuple(shape):
        raise MrfError(f"{name} must have shape {tuple(shape)}, got {tuple(t.shape)}")
    if dtype is not None and t.dtype != dtype:
        raise MrfError(f"{name} must be {dtype}, got {t.dtype}")
    if device is not None and t.device != device:
        raise MrfError(f"{name} must live on {device}, got {t.device}")
    if not t.is_contiguous():
        raise MrfError(f"{name} must be contiguous")
    return t


def _chk_np(name, a, shape, dtype):
    """Caller-supplied numpy output buffers of the host entries."""
    if a is None:
        return None
    if not isinstance(a, np.ndarray) or a.dtype != dtype or tuple(a.shape) != tuple(shape) or not a.flags.c_contiguous:
        raise MrfError(f"{name} must be a C-contiguous {np.dtype(dtype).name} array of shape {tuple(shape)}")
    return a


class Fabrics:
    """One planner configuration (MrfConfig) on one B200."""

    def __init__(self, n_robots: int = 2, device: int = 0, config=None, **overrides):
        self.cfg = config if config is not None else default_config(n_robots, **overrides)
        self.n_robots = int(self.cfg.n_robots)
        self.device = device
        self.handle = Handle(self.cfg, device)

    def close(self):
        self.handle.close()

    # ------------------------------------------------------------------ host buffers (AoS)
    def rollout_host(self, rec, N: int, dtype: str = "f64", trajectories: bool = False, out=None):
        """rec (B,R,44) -> dict(avg_vel (B,R), x_ee (B,R,3), goal_est (B,3)[, qN, qdN (B,R,N,7)])."""
        dt = _NP[dtype]
        R = self.n_robots
        rec = np.ascontiguousarray(rec, dtype=dt)
        if rec.ndim == 2:
            rec = rec[None]
        if rec.shape[1:] != (R, REC):
            raise MrfError(f"rec must be (B,{R},{REC}), got {rec.shape}")
        B = rec.shape[0]
        o = out if out is not None else {}
        o.setdefault("avg_vel", np.empty((B, R), dt))
        o.setdefault("x_ee", np.empty((B, R, 3), dt))
        o.setdefault("goal_est", np.empty((B, 3), dt))
        if trajectories:
            o.setdefault("qN", np.empty((B, R, N, DOF), dt))
            o.setdefault("qdN", np.empty((B, R, N, DOF), dt))
        for k, shp in (("avg_vel", (B, R)), ("x_ee", (B, R, 3)), ("goal_est", (B, 3)), ("qN", (B, R, N, DOF)),
                       ("qdN", (B, R, N, DOF))):
            _chk_np(k, o.get(k), shp, dt)
        fn = getattr(lib(), f"mrf_rollout_host_{dtype}")
        check(fn(self.handle.ptr, hptr(rec), N, hptr(o["avg_vel"]), hptr(o["x_ee"]), hptr(o["goal_est"]),
                 hptr(o.get("qN")), hptr(o.get("qdN")), B), "mrf_rollout_host")
        return o

    def rollout_host_submit(self, rec, N: int, out: dict, dtype: str = "f32", shared=None):
        """Asynchronous rollout_host for sweeps: `rec` (B,R,44) and the arrays in `out` (avg_vel (B,R), x_ee (B,R,3),
        goal_est (B,3); any subset) must be page-locked numpy arrays of the entry's dtype and stay untouched until
        rollout_host_wait().  Up to two batches are in flight."""
        dt = _NP[dtype]
        R = self.n_robots
        if rec.ndim != 3:
            raise MrfError(f"rollout_host_submit: rec must be (B,{R},F), got {rec.shape}")
        B = rec.shape[0]
        _chk_np("rec", rec, (B, R, 18 if shared is not None else REC), dt)
        for k, shp in (("avg_vel", (B, R)), ("x_ee", (B, R, 3)), ("goal_est", (B, 3))):
            _chk_np(k, out.get(k), shp, dt)
        if set(out) - {"avg_vel", "x_ee", "goal_est"}:
            raise MrfError("rollout_host_submit: out takes avg_vel, x_ee, goal_est only")
        if shared is not None:     # compact records: rec (B,R,18) = q, qdot, x_goal_0, weight_goal_0; shared (R,44)
            shared = np.ascontiguousarray(shared, dtype=dt).reshape(self.n_robots, REC)
            fn = getattr(lib(), f"mrf_rollout_host_submit_compact_{dtype}")
            check(fn(self.handle.ptr, hptr(rec), hptr(shared), N, hptr(out.get("avg_vel")), hptr(out.get("x_ee")),
                     hptr(out.get("goal_est")), rec.shape[0]), "mrf_rollout_host_submit_compact")
            return
        fn = getattr(lib(), f"mrf_rollout_host_submit_{dtype}")
        check(fn(self.handle.ptr, hptr(rec), N, hptr(out.get("avg_vel")), hptr(out.get("x_ee")), hptr(out.get("goal_est")),
                 rec.shape[0]), "mrf_rollout_host_submit")

    def rfcv_host_submit(self, rec, N: int, result, shared=None, time_step: int = 100, goals_out=None):
        """One whole RF-CV step of a sweep from host memory (mrf_rfcv_host_submit_f32): page-locked float32 records
        rec (B,R,44) -- or compact (B,R,18) with shared (R,44) -- -> page-locked result (R+1,B): avg_vel rows + deadlock
        flag; goals_out (4,R,B) optional.  Asynchronous: rollout_host_wait() before reading the results."""
        R = self.n_robots
        if rec.ndim != 3:
            raise MrfError(f"rfcv_host_submit: rec must be (B,{R},F), got {rec.shape}")
        B = rec.shape[0]
        _chk_np("rec", rec, (B, R, 18 if shared is not None else REC), np.float32)
        _chk_np("result", result, (R + 1, B), np.float32)
        _chk_np("goals_out", goals_out, (4, R, B), np.float32)
        if shared is not None:
            shared = np.ascontiguousarray(shared, dtype=np.float32).reshape(R, REC)
        check(lib().mrf_rfcv_host_submit_f32(self.handle.ptr, hptr(rec), hptr(shared), N, int(time_step), hptr(result),
                                             hptr(goals_out), B), "mrf_rfcv_host_submit")

    def rollout_host_wait(self, all: bool = False):
        check(lib().mrf_rollout_host_wait(self.handle.ptr, 1 if all else 0), "mrf_rollout_host_wait")

    def action_host(self, rec, obst=None, robot_first: int = 0, dtype: str = "f64"):
        """rec (B,n_rob,44), obst (B,n_rob,S,10) -> action (B,n_rob,7)."""
        dt = _NP[dtype]
        rec = np.ascontiguousarray(rec, dtype=dt)
        if rec.ndim == 2:
            rec = rec[:, None, :]
        B, n_rob = rec.shape[0], rec.shape[1]
        if obst is None:
            S, obst_a = 0, None
        else:
            obst_a = np.ascontiguousarray(obst, dtype=dt).reshape(B, n_rob, -1, OBST)
            S = obst_a.shape[2]
            if S == 0:
                obst_a = None
        act = np.empty((B, n_rob, DOF), dt)
        fn = getattr(lib(), f"mrf_action_host_{dtype}")
        check(fn(self.handle.ptr, robot_first, n_rob, hptr(rec), S, hptr(obst_a), hptr(act), B), "mrf_action_host")
        return act

    def rollout_cart_host(self, robot: int, rec, obst, N: int, dtype: str = "f64", trajectories: bool = True):
        """rec (B,44), obst (B,S,10) -> avg_vel (B,), qN, qdN (B,N,7)."""
        dt = _NP[dtype]
        rec = np.ascontiguousarray(rec, dtype=dt).reshape(-1, REC)
        B = rec.shape[0]
        obst_a = np.ascontiguousarray(obst, dtype=dt).reshape(B, -1, OBST)
        S = obst_a.shape[1]
        avg = np.empty((B,), dt)
        qN = np.empty((B, N, DOF), dt) if trajectories else None
        qdN = np.empty((B, N, DOF), dt) if trajectories else None
        fn = getattr(lib(), f"mrf_rollout_cart_host_{dtype}")
        check(fn(self.handle.ptr, robot, hptr(rec), S, hptr(obst_a if S else None), N, hptr(avg), hptr(qN), hptr(qdN), B),
              "mrf_rollout_cart_host")
        return avg, qN, qdN

    def kinematics_host(self, q, qdot):
        """q, qdot (B,R,7) -> x, v, a (B,R,8,3); a = jdot_ref_sign * d(J qdot)/dq qdot (utils.py:28,37)."""
        R = self.n_robots
        q = np.ascontiguousarray(q, dtype=np.float64).reshape(-1, R, DOF)
        qd = np.ascontiguousarray(qdot, dtype=np.float64).reshape(-1, R, DOF)
        B = q.shape[0]
        x, v, a = (np.empty((B, R, NLINKS, 3)) for _ in range(3))
        check(lib().mrf_kinematics_host_f64(self.handle.ptr, hptr(q), hptr(qd), hptr(x), hptr(v), hptr(a), B),
              "mrf_kinematics_host")
        return x, v, a

    # ------------------------------------------------------------------ device tensors (SoA)
    @staticmethod
    def _tp(t):
        return None if t is None else C.c_void_p(t.data_ptr())

    @staticmethod
    def _prec(t):
        import torch
        if t.dtype == torch.float64:
            return "f64"
        if t.dtype == torch.float32:
            return "f32"
        raise MrfError(f"unsupported dtype {t.dtype}")

    def _stream(self):
        import torch
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def rollout_dev(self, rec, N: int, avg_vel=None, x_ee=None, goal_est=None, qN=None, qdN=None, risk=None):
        """rec: torch (44,R,B) on this device; outputs as in include/mrf_b200.h (allocated if None for avg_vel).
        risk (R,B): also return the stiffness indicator (mrf_rollout_risk_dev, no trajectories)."""
        import torch
        p = self._prec(rec)
        if rec.dim() != 3:
            raise MrfError("rec must be a contiguous (44,R,B) tensor")
        _, R, B = rec.shape
        if R != self.n_robots:
            raise MrfError(f"rec must be (44,{self.n_robots},B), got {tuple(rec.shape)}")
        _chk("rec", rec, (REC, R, B), optional=False)
        dt, dev = rec.dtype, rec.device
        if avg_vel is None:
            avg_vel = torch.empty((R, B), dtype=dt, device=dev)
        _chk("avg_vel", avg_vel, (R, B), dt, dev)
        _chk("x_ee", x_ee, (R, 3, B), dt, dev)
        _chk("goal_est", goal_est, (3, B), dt, dev)
        _chk("qN", qN, (R, N, DOF, B), dt, dev)
        _chk("qdN", qdN, (R, N, DOF, B), dt, dev)
        if risk is not None:
            if qN is not None or qdN is not None:
                raise MrfError("rollout_dev: risk and trajectory outputs are separate entries")
            _chk("risk", risk, (R, B), dt, dev)
            fn = getattr(lib(), f"mrf_rollout_risk_dev_{p}")
            check(fn(self.handle.ptr, self._tp(rec), N, self._tp(avg_vel), self._tp(x_ee), self._tp(goal_est),
                     self._tp(risk), B, self._stream()), "mrf_rollout_risk_dev")
            return avg_vel
        fn = getattr(lib(), f"mrf_rollout_dev_{p}")
        check(fn(self.handle.ptr, self._tp(rec), N, self._tp(avg_vel), self._tp(x_ee), self._tp(goal_est), self._tp(qN),
                 self._tp(qdN), B, self._stream()), "mrf_rollout_dev")
        return avg_vel

    def rollout_static_dev(self, rec, stat, N: int, avg_vel=None, x_ee=None, goal_est=None, qN=None, qdN=None):
        """Coupled rollout with static spheres per robot: rec (44,R,B), stat (S,4,R,B) = x, y, z, radius
        (mrf_rollout_static_dev; forward_planner_Jointspace.py:319-322)."""
        import torch
        p = self._prec(rec)
        _, R, B = rec.shape
        dt, dev = rec.dtype, rec.device
        _chk("rec", rec, (REC, self.n_robots, B), optional=False)
        S = 0 if stat is None else stat.shape[0]
        _chk("stat", stat, (S, 4, R, B), dt, dev)
        if avg_vel is None:
            avg_vel = torch.empty((R, B), dtype=dt, device=dev)
        _chk("avg_vel", avg_vel, (R, B), dt, dev)
        _chk("x_ee", x_ee, (R, 3, B), dt, dev)
        _chk("goal_est", goal_est, (3, B), dt, dev)
        _chk("qN", qN, (R, N, DOF, B), dt, dev)
        _chk("qdN", qdN, (R, N, DOF, B), dt, dev)
        fn = getattr(lib(), f"mrf_rollout_static_dev_{p}")
        check(fn(self.handle.ptr, self._tp(rec), N, S, self._tp(stat), self._tp(avg_vel), self._tp(x_ee), self._tp(goal_est),
                 self._tp(qN), self._tp(qdN), B, self._stream()), "mrf_rollout_static_dev")
        return avg_vel

    def rfcv_post_dev(self, rec, N: int, x_ee, rec_work, goal_est, avg_vel, sm_state, time_step, time_deadlock_out, st_int,
                      st_goal, risk=None, flag=None, result=None, slot: int = 0):
        """Post step of an RF-CV sweep (mrf_rfcv_post_dev): deadlock heuristic in place on rec_work, per-scenario results
        into result (R+1,B); FP32 with `risk`: guard-band / stiff scenarios are re-rolled in FP64 first so that the flags
        equal a float64 evaluation of the same records.  Post steps that may run concurrently (different streams) need
        different scratch slots (0..3)."""
        import torch
        p = self._prec(rec)
        _, R, B = rec.shape
        dt, dev, i32 = rec.dtype, rec.device, torch.int32
        _chk("rec", rec, (REC, self.n_robots, B), dt, dev, optional=False)
        _chk("rec_work", rec_work, (REC, R, B), dt, dev, optional=False)
        _chk("x_ee", x_ee, (R, 3, B), dt, dev, optional=False)
        _chk("avg_vel", avg_vel, (R, B), dt, dev, optional=False)
        _chk("goal_est", goal_est, (3, B), dt, dev)
        _chk("risk", risk, (R, B), dt, dev)
        _chk("sm_state", sm_state, (R, B), i32, dev, optional=False)
        _chk("time_step", time_step, (B,), i32, dev, optional=False)
        _chk("time_deadlock_out", time_deadlock_out, (B,), i32, dev, optional=False)
        _chk("st_int", st_int, (4 * B,), i32, dev, optional=False)
        _chk("st_goal", st_goal, (3, B), dt, dev, optional=False)
        if flag is None:
            flag = torch.empty((B,), dtype=i32, device=dev)
        _chk("flag", flag, (B,), i32, dev)
        _chk("result", result, (R + 1, B), dt, dev)
        fn = getattr(lib(), f"mrf_rfcv_post_dev_{p}")
        check(fn(self.handle.ptr, self._tp(rec), N, self._tp(x_ee), self._tp(rec_work), self._tp(goal_est),
                 self._tp(avg_vel), self._tp(risk), self._tp(sm_state), self._tp(time_step), self._tp(time_deadlock_out),
                 self._tp(st_int), self._tp(st_goal), self._tp(flag), self._tp(result), B, self._stream(), int(slot)),
              "mrf_rfcv_post_dev")
        return flag

    def set_guard(self, bands=None, risk_edges=None, band_dist=-1.0, cap=-1):
        """mrf_set_guard: bands (6,) = absolute then relative band per tier, risk_edges (2,); None / negative = keep."""
        b = None if bands is None else (C.c_double * 6)(*[float(v) for v in bands])
        e = None if risk_edges is None else (C.c_double * 2)(*[float(v) for v in risk_edges])
        check(lib().mrf_set_guard(self.handle.ptr, b, e, band_dist, cap), "mrf_set_guard")

    def guard_stats(self):
        """(re-rolled so far, overflow so far, listed by the last call); synchronise first."""
        out = (C.c_int64 * 3)()
        check(lib().mrf_guard_stats(self.handle.ptr, out), "mrf_guard_stats")
        return int(out[0]), int(out[1]), int(out[2])

    def action_dev(self, rec, obst, action=None, robot_first: int = 0):
        """rec (44,n_rob,B), obst (S,10,n_rob,B) or None -> action (7,n_rob,B)."""
        import torch
        p = self._prec(rec)
        if rec.dim() != 3:
            raise MrfError("rec must be a contiguous (44,n_rob,B) tensor")
        _, n_rob, B = rec.shape
        dt, dev = rec.dtype, rec.device
        _chk("rec", rec, (REC, n_rob, B), optional=False)
        S = 0 if obst is None else obst.shape[0]
        _chk("obst", obst, (S, OBST, n_rob, B), dt, dev)
        if action is None:
            action = torch.empty((DOF, n_rob, B), dtype=dt, device=dev)
        _chk("action", action, (DOF, n_rob, B), dt, dev)
        fn = getattr(lib(), f"mrf_action_dev_{p}")
        check(fn(self.handle.ptr, robot_first, n_rob, self._tp(rec), S, self._tp(obst), self._tp(action), B,
                 self._stream()), "mrf_action_dev")
        return action

    def rollout_cart_dev(self, robot: int, rec, obst, N: int, avg_vel=None, qN=None, qdN=None):
        import torch
        p = self._prec(rec)
        B = rec.shape[-1]
        dt, dev = rec.dtype, rec.device
        if rec.dim() == 3:
            _chk("rec", rec, (REC, 1, B), optional=False)
        else:
            _chk("rec", rec, (REC, B), optional=False)
        S = 0 if obst is None else obst.shape[0]
        if obst is not None:
            _chk("obst", obst, (S, OBST, 1, B) if obst.dim() == 4 else (S, OBST, B), dt, dev)
        if avg_vel is None:
            avg_vel = torch.empty((B,), dtype=dt, device=dev)
        _chk("avg_vel", avg_vel, (B,), dt, dev)
        _chk("qN", qN, (N, DOF, B), dt, dev)
        _chk("qdN", qdN, (N, DOF, B), dt, dev)
        fn = getattr(lib(), f"mrf_rollout_cart_dev_{p}")
        check(fn(self.handle.ptr, robot, self._tp(rec), S, self._tp(obst), N, self._tp(avg_vel), self._tp(qN),
                 self._tp(qdN), B, self._stream()), "mrf_rollout_cart_dev")
        return avg_vel

    def rollout_cart_all_dev(self, rec, obst, N: int, avg_vel=None, qN=None, qdN=None):
        """Cartesian rollouts of every robot in one launch (mrf_rollout_cart_all_dev): rec (44,R,B), obst (S,10,R,B) or
        None -> avg_vel (R,B); qN, qdN (R,N,7,B) optional.  Robot r's results equal rollout_cart_dev(r, ...) on its slices."""
        import torch
        p = self._prec(rec)
        R = self.n_robots
        if rec.dim() != 3:
            raise MrfError(f"rec must be a contiguous (44,{R},B) tensor")
        B = rec.shape[-1]
        dt, dev = rec.dtype, rec.device
        _chk("rec", rec, (REC, R, B), optional=False)
        S = 0 if obst is None else obst.shape[0]
        _chk("obst", obst, (S, OBST, R, B), dt, dev)
        if avg_vel is None:
            avg_vel = torch.empty((R, B), dtype=dt, device=dev)
        _chk("avg_vel", avg_vel, (R, B), dt, dev)
        _chk("qN", qN, (R, N, DOF, B), dt, dev)
        _chk("qdN", qdN, (R, N, DOF, B), dt, dev)
        fn = getattr(lib(), f"mrf_rollout_cart_all_dev_{p}")
        check(fn(self.handle.ptr, self._tp(rec), S, self._tp(obst), N, self._tp(avg_vel), self._tp(qN), self._tp(qdN), B,
                 self._stream()), "mrf_rollout_cart_all_dev")
        return avg_vel

    def kinematics_dev(self, q, qdot, x=None, v=None, a=None):
        import torch
        p = self._prec(q)
        _, R, B = q.shape
        dt, dev = q.dtype, q.device
        _chk("q", q, (DOF, self.n_robots, B), optional=False)
        _chk("qdot", qdot, (DOF, R, B), dt, dev, optional=False)
        mk = lambda: torch.empty((NLINKS, 3, R, B), dtype=dt, device=dev)
        x = mk() if x is None else x
        v = mk() if v is None else v
        a = mk() if a is None else a
        for n_, t_ in (("x", x), ("v", v), ("a", a)):
            _chk(n_, t_, (NLINKS, 3, R, B), dt, dev)
        fn = getattr(lib(), f"mrf_kinematics_dev_{p}")
        check(fn(self.handle.ptr, self._tp(q), self._tp(qdot), self._tp(x), self._tp(v), self._tp(a), B, self._stream()),
              "mrf_kinematics_dev")
        return x, v, a

    def obstacles_dev(self, q, qdot, n_per_link: int = 1, vel_mode: int = 0, offsets=None, obst=None, spheres_x=None,
                      spheres_v=None, want_obst: bool = True):
        """q, qdot (7,R,B) -> obst (8 n (R-1), 10, R, B): the other robots' collision spheres of every ego robot."""
        import torch
        from .spheres import sphere_offsets
        p = self._prec(q)
        _, R, B = q.shape
        dt, dev = q.dtype, q.device
        _chk("q", q, (DOF, self.n_robots, B), optional=False)
        _chk("qdot", qdot, (DOF, R, B), dt, dev, optional=False)
        off = np.ascontiguousarray(sphere_offsets(n_per_link) if offsets is None else offsets, dtype=np.float64)
        if off.shape != (NLINKS, n_per_link, 3):
            raise MrfError(f"offsets must be ({NLINKS},{n_per_link},3), got {off.shape}")
        if want_obst and obst is None:
            obst = torch.empty((8 * n_per_link * (R - 1), OBST, R, B), dtype=dt, device=dev)
        _chk("obst", obst, (8 * n_per_link * (R - 1), OBST, R, B), dt, dev)
        _chk("spheres_x", spheres_x, (8 * n_per_link, 3, R, B), dt, dev)
        _chk("spheres_v", spheres_v, (8 * n_per_link, 3, R, B), dt, dev)
        fn = getattr(lib(), f"mrf_obstacles_dev_{p}")
        check(fn(self.handle.ptr, n_per_link, hptr(off), vel_mode, self._tp(q), self._tp(qdot), self._tp(obst),
                 self._tp(spheres_x), self._tp(spheres_v), B, self._stream()), "mrf_obstacles_dev")
        return obst

    def point_action_dev(self, rec, stat=None, dyn=None, action=None):
        """Point-mass planner (config C1): rec (10,B), stat (Ss,4,B), dyn (Sd,7,B) -> action (3,B)."""
        import torch
        p = self._prec(rec)
        B = rec.shape[-1]
        dt, dev = rec.dtype, rec.device
        _chk("rec", rec, (10, B), optional=False)
        _chk("stat", stat, (0 if stat is None else stat.shape[0], 4, B), dt, dev)
        _chk("dyn", dyn, (0 if dyn is None else dyn.shape[0], 7, B), dt, dev)
        if action is None:
            action = torch.empty((3, B), dtype=dt, device=dev)
        _chk("action", action, (3, B), dt, dev)
        fn = getattr(lib(), f"mrf_point_action_dev_{p}")
        check(fn(self.handle.ptr, self._tp(rec), 0 if stat is None else stat.shape[0], self._tp(stat),
                 0 if dyn is None else dyn.shape[0], self._tp(dyn), self._tp(action), B, self._stream()),
              "mrf_point_action_dev")
        return action

    def deadlock_dev(self, x_ee, goals, weights, sm_state, time_step, time_deadlock_out, st_int, st_goal,
                     avg_vel=None, avg_sum=None, flag=None):
        """Batched deadlock_checking step; goals/weights/time_deadlock_out/st_* are updated in place.
        Give avg_vel (R,B) (per-robot rollout averages) or avg_sum (B,)."""
        import torch
        p = self._prec(x_ee)
        R, B = self.n_robots, x_ee.shape[-1]
        dt, dev, i32 = x_ee.dtype, x_ee.device, torch.int32
        _chk("x_ee", x_ee, (R, 3, B), optional=False)
        _chk("goals", goals, (R, 3, B), dt, dev, optional=False)
        _chk("weights", weights, (R, B), dt, dev, optional=False)
        self._chk_dl_state(sm_state, time_step, time_deadlock_out, st_int, st_goal, R, B, dt, dev)
        _chk("avg_vel", avg_vel, (R, B), dt, dev)
        _chk("avg_sum", avg_sum, (B,), dt, dev)
        if flag is None:
            flag = torch.empty((B,), dtype=i32, device=dev)
        _chk("flag", flag, (B,), i32, dev)
        fn = getattr(lib(), f"mrf_deadlock_dev_{p}")
        check(fn(self.handle.ptr, self._tp(x_ee), self._tp(goals), self._tp(weights), self._tp(avg_vel),
                 self._tp(avg_sum), self._tp(sm_state), self._tp(time_step), self._tp(time_deadlock_out), self._tp(st_int),
                 self._tp(st_goal), self._tp(flag), B, self._stream()), "mrf_deadlock_dev")
        return flag

    @staticmethod
    def _chk_dl_state(sm_state, time_step, time_deadlock_out, st_int, st_goal, R, B, dt, dev):
        import torch
        i32 = torch.int32
        _chk("sm_state", sm_state, (R, B), i32, dev, optional=False)
        _chk("time_step", time_step, (B,), i32, dev, optional=False)
        _chk("time_deadlock_out", time_deadlock_out, (B,), i32, dev, optional=False)
        if st_int is None or st_int.numel() != 4 * B:
            raise MrfError(f"st_int must hold 4 x {B} int32")
        _chk("st_int", st_int, tuple(st_int.shape), i32, dev, optional=False)
        _chk("st_goal", st_goal, (3, B), dt, dev, optional=False)


def _deadlock_rec_dev(self, x_ee, rec, sm_state, time_step, time_deadlock_out, st_int, st_goal, goal_est=None, avg_vel=None,
                      avg_sum=None, flag=None):
    """deadlock_checking in place on the record tensor (goal rows 14..16, weight row 17); see mrf_deadlock_rec_dev."""
    import torch
    p = self._prec(rec)
    R, B = self.n_robots, rec.shape[-1]
    dt, dev = rec.dtype, rec.device
    _chk("rec", rec, (REC, R, B), optional=False)
    _chk("x_ee", x_ee, (R, 3, B), dt, dev, optional=False)
    self._chk_dl_state(sm_state, time_step, time_deadlock_out, st_int, st_goal, R, B, dt, dev)
    _chk("goal_est", goal_est, (3, B), dt, dev)
    _chk("avg_vel", avg_vel, (R, B), dt, dev)
    _chk("avg_sum", avg_sum, (B,), dt, dev)
    if flag is None:
        flag = torch.empty((B,), dtype=torch.int32, device=dev)
    _chk("flag", flag, (B,), torch.int32, dev)
    fn = getattr(lib(), f"mrf_deadlock_rec_dev_{p}")
    check(fn(self.handle.ptr, self._tp(x_ee), self._tp(rec), self._tp(goal_est), self._tp(avg_vel), self._tp(avg_sum),
             self._tp(sm_state), self._tp(time_step), self._tp(time_deadlock_out), self._tp(st_int), self._tp(st_goal),
             self._tp(flag), B, self._stream()), "mrf_deadlock_rec_dev")
    return flag


Fabrics.deadlock_rec_dev = _deadlock_rec_dev


def _fsm_dev(self, nr_blocks, x_ee, q_grip, goal_block, start_goal, goal, above, weight, st, grip_action=None):
    """Batched pick-and-place state machine step (state_machine.py:133-214); goal/above/weight/st updated in place."""
    import torch
    p = self._prec(x_ee)
    R, B = self.n_robots, x_ee.shape[-1]
    dt, dev = x_ee.dtype, x_ee.device
    nb = np.ascontiguousarray(nr_blocks, dtype=np.int32)
    if nb.shape != (R,):
        raise MrfError(f"nr_blocks must hold {R} integers")
    for n_, t_ in (("x_ee", x_ee), ("goal_block", goal_block), ("start_goal", start_goal), ("goal", goal), ("above", above)):
        _chk(n_, t_, (R, 3, B), dt, dev, optional=False)
    _chk("q_grip", q_grip, (R, 2, B), dt, dev, optional=False)
    _chk("weight", weight, (R, B), dt, dev, optional=False)
    _chk("st", st, (6, R, B), torch.int32, dev, optional=False)
    _chk("grip_action", grip_action, (R, 2, B), dt, dev)
    fn = getattr(lib(), f"mrf_fsm_dev_{p}")
    check(fn(self.handle.ptr, hptr(nb), self._tp(x_ee), self._tp(q_grip), self._tp(goal_block), self._tp(start_goal),
             self._tp(goal), self._tp(above), self._tp(weight), self._tp(st), self._tp(grip_action), B, self._stream()),
          "mrf_fsm_dev")


Fabrics.fsm_dev = _fsm_dev


def to_soa(rec):
    """(B,R,F) array-of-records -> (F,R,B) structure-of-arrays (numpy or torch)."""
    if isinstance(rec, np.ndarray):
        return np.ascontiguousarray(rec.transpose(2, 1, 0))
    return rec.permute(2, 1, 0).contiguous()
