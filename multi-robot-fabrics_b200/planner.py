"""The reference's planner call surface on top of the CUDA hot path (drop-in for that path only).

Mirrors, with the same names, argument meaning and return shapes:
  set_planner_panda(...) -> (planner, goal)      examples/example_pandas_Jointspace.py:64-134
  planner.compute_action(**kwargs)               fabrics ParameterizedFabricPlanner.compute_action as called at
                                                 examples/example_pandas_Jointspace.py:417-445,
                                                 forward_planner_Cartesian.py:150-190
  ForwardFabricsPlanner                          multi_robot_fabrics/fabrics_planner/forward_planner_Jointspace.py:12-423
  FabricsRollouts                                multi_robot_fabrics/fabrics_planner/forward_planner_Cartesian.py:8-563
  deadlockprevention                             multi_robot_fabrics/others_planner/deadlock_prevention.py:4-118

What cannot be reproduced: ``planner._funs._function(*SX)`` symbolic inlining (forward_planner_Jointspace.py:185,233);
the rollout classes here subsume the whole horizon instead, so ``forward_multi_fabrics_symbolic()`` /
``symbolic_forward_fabrics()`` are cheap set-up steps.  Every number is computed by libmrf_b200.so on the GPU; if the
library or a B200 is missing the constructors raise MrfError (no CPU fallback).
"""
from __future__ import annotations

import math
import warnings

import numpy as np

from ._lib import ANG, CON, DOF, G0, G1, G2, MAX_SELF_PAIRS, OBST, Q, QD, RB, REC, W0, W1, W2, MrfError, check, default_config, hptr, lib
from .api import Fabrics

PANDA_LIMITS = [[-2.8973, 2.8973], [-1.7628, 1.7628], [-2.8973, 2.8973], [-3.0718, -0.0698],
                [-2.8973, 2.8973], [-0.0175, 3.7525], [-2.8973, 2.8973]]
ROT_PANDA = np.array([[0.0, 0.0, -1.0], [0.0, 1.0, 0.0], [1.0, 0.0, 0.0]])


def _vec(v, n=None):
    a = np.asarray(v, dtype=np.float64).reshape(-1)
    if n is not None and a.size != n:
        raise MrfError(f"expected {n} values, got {a.size}")
    return a


def mount_transform(i_robot: int, mount_param: dict) -> np.ndarray:
    """examples/example_pandas_Jointspace.py:108-118."""
    angle = math.pi if i_robot in (1, 2) else 0.0
    T = np.identity(4)
    T[0:2, 0:2] = np.array([[np.cos(angle), -np.sin(angle)], [np.sin(angle), np.cos(angle)]])
    T[0:3, 3] = mount_param["mount_positions"][i_robot]
    return T


class _SubGoal:
    def __init__(self, weight, desired_position):
        self.weight = weight
        self.desired_position = desired_position


class _GoalConfig:
    def __init__(self):
        self.subgoal0 = _SubGoal(2.0, [0.1, 0.6, 0.8])
        self.subgoal1 = _SubGoal(10.0, [0.107, 0.0, 0.0])
        self.subgoal2 = _SubGoal(1.0, [np.pi / 4])

    def __len__(self):
        return 3


class PandaGoal:
    """Stand-in for the GoalComposition of create_dummy_goal_panda (example_pandas_Jointspace.py:25-62): only the
    attributes the rollout classes read (``_config.subgoalN.{weight,desired_position}``, ``len(_config)``)."""

    def __init__(self):
        self._config = _GoalConfig()


def _link_number(name) -> int:
    """'panda_linkN' -> N, 'panda_hand' -> 9 (the numbering of mrf_set_self_collision)."""
    if name == "panda_hand":
        return 9
    if isinstance(name, str) and name.startswith("panda_link") and name[len("panda_link"):].isdigit():
        n = int(name[len("panda_link"):])
        if 1 <= n <= 8:
            return n
    raise MrfError(f"self-collision link must be panda_link1..8 or panda_hand, got {name!r}")


def self_collision_pair_list(pairs: dict):
    """fabrics' self_collision_pairs dict {link: [paired links]} -> [(a, b)] link numbers, each unordered pair once.
    Pairs whose two points coincide identically ((a, a), link5/link6, link8/panda_hand, both in link1/link2) have the leaf
    0/0; fabrics skips such a pair with a warning and so does this."""
    out = []
    for a_name, others in (pairs or {}).items():
        a = _link_number(a_name)
        for b_name in others:
            b = _link_number(b_name)
            lo, hi = min(a, b), max(a, b)
            if lo == hi or (lo, hi) in ((5, 6), (8, 9)) or hi <= 2:
                warnings.warn(f"self-collision pair ({a_name}, {b_name}): the two points coincide, pair skipped")
                continue
            if (lo, hi) not in [(min(x), max(x)) for x in out]:
                out.append((a, b))
    if len(out) > MAX_SELF_PAIRS:
        raise MrfError(f"at most {MAX_SELF_PAIRS} self-collision pairs per robot, got {len(out)}")
    return out


class PandaFabricPlanner:
    """compute_action drop-in for the planner built by set_planner_panda."""

    def __init__(self, mount: np.ndarray, nr_obst: int, nr_obst_dyn: int, collision_links_nr, i_robot: int = 0,
                 device: int = 0, limits=PANDA_LIMITS, mode: str = "vel", time_step: float = 0.01, dtype: str = "f64",
                 self_collision_pairs=None):
        self.mount = np.asarray(mount, dtype=np.float64).reshape(4, 4)
        self.self_pairs = self_collision_pair_list(self_collision_pairs)
        self.self_rho = None               # rho of each pair as last set on the handle (from compute_action's radii)
        self.i_robot = i_robot
        self.nr_obst, self.nr_obst_dyn = int(nr_obst), int(nr_obst_dyn)
        # Any subset of panda_link1..8 (the reference's signature default is [5]); links with constant fk (panda_link1/2)
        # carry no leaves, an empty list is the grasp planner.  Numbers >= 9 mean 'panda_hand'
        # (example_pandas_Jointspace.py:91-96), whose origin is panda_link8's: accepted in place of link 8 only.
        links = [int(l) for l in collision_links_nr]
        if any(l >= 9 for l in links):
            if 8 in links:
                raise MrfError("panda_hand next to panda_link8 (two leaves at one point) is not implemented")
            links = [min(l, 8) for l in links]
        if any(l < 1 for l in links):
            raise MrfError(f"collision_links_nr must be link numbers >= 1, got {collision_links_nr}")
        self.collision_links_all = sorted(set(links))
        self.collision_links_nr = [l for l in self.collision_links_all if l > 2]
        self.dtype = dtype
        cfg = default_config(1, mode=1 if mode == "vel" else 0, dt=time_step,
                             has_collision_links=1 if self.collision_links_nr else 0, mount=[self.mount], limits=limits,
                             collision_links=[self.collision_links_all])
        self.fab = Fabrics(config=cfg, device=device)

    # fabrics' CasadiFunctionWrapper expands list / dict kwargs into per-index parameters
    def _record_and_obstacles(self, kw: dict):
        rec = np.zeros(REC)
        rec[Q:Q + 7] = _vec(kw["q"], 7)
        rec[QD:QD + 7] = _vec(kw["qdot"], 7)
        rec[G0:G0 + 3] = _vec(kw["x_goal_0"], 3)
        rec[W0] = float(np.asarray(kw["weight_goal_0"]).reshape(-1)[0])
        rec[G1:G1 + 3] = _vec(kw.get("x_goal_1", [0.107, 0.0, 0.0]), 3)
        rec[W1] = float(np.asarray(kw.get("weight_goal_1", 0.0)).reshape(-1)[0])
        rec[G2] = _vec(kw.get("x_goal_2", [0.0]))[0]
        rec[W2] = float(np.asarray(kw.get("weight_goal_2", 0.0)).reshape(-1)[0])
        rec[ANG:ANG + 9] = np.asarray(kw.get("angle_goal_1", ROT_PANDA), dtype=np.float64).reshape(9)
        rec[CON:CON + 4] = _vec(kw.get("constraint_0", [0.0, 0.0, 1.0, 0.0]), 4)
        links = kw.get("radius_body_panda_links", {})
        for i, l in enumerate(range(3, 9)):
            key = f"radius_body_panda_link{l}"
            if key in kw:
                rec[RB + i] = float(np.asarray(kw[key]).reshape(-1)[0])
            elif str(l) in links:
                rec[RB + i] = float(np.asarray(links[str(l)]).reshape(-1)[0])
            elif l in links:
                rec[RB + i] = float(np.asarray(links[l]).reshape(-1)[0])
            elif l in self.collision_links_nr:
                raise KeyError(key)        # a collision link needs its radius_body parameter, as in fabrics
        if not self.collision_links_nr:
            # no collision links -> fabrics creates no obstacle leaves, so no obstacle parameter exists in the function
            # (the grasp planner is built with nr_obst = nr_obst_dyn = i_robot, example_pandas_Jointspace.py:160-166)
            return rec, np.zeros((0, OBST))
        obst = np.zeros((self.nr_obst + self.nr_obst_dyn, OBST))
        for i in range(self.nr_obst):                      # static spheres: x_obst_i, radius_obst_i
            x = kw[f"x_obst_{i}"] if f"x_obst_{i}" in kw else kw["x_obsts"][i]
            r = kw[f"radius_obst_{i}"] if f"radius_obst_{i}" in kw else kw["radius_obsts"][i]
            obst[i, 0:3] = _vec(x, 3)
            obst[i, 9] = float(np.asarray(r).reshape(-1)[0])
        for i in range(self.nr_obst_dyn):                  # dynamic spheres
            o = self.nr_obst + i
            get = lambda single, plural: kw[f"{single}_{i}"] if f"{single}_{i}" in kw else kw[plural][i]
            obst[o, 0:3] = _vec(get("x_obst_dynamic", "x_obsts_dynamic"), 3)
            obst[o, 3:6] = _vec(get("xdot_obst_dynamic", "xdot_obsts_dynamic"), 3)
            obst[o, 6:9] = _vec(get("xddot_obst_dynamic", "xddot_obsts_dynamic"), 3)
            obst[o, 9] = float(np.asarray(get("radius_obst_dynamic", "radius_obsts_dynamic")).reshape(-1)[0])
        return rec, obst

    def _self_collision_radii(self, kw: dict):
        """rho = r_a + r_b of each pair from the radii the reference passes: radius_body_panda_links[str(l)] (or
        radius_body_panda_link{l}) and radius_body_panda_hand."""
        links = kw.get("radius_body_panda_links", {})

        def radius(l):
            if l == 9:
                if "radius_body_panda_hand" not in kw:
                    raise MrfError("self-collision pair with panda_hand needs radius_body_panda_hand")
                return float(np.asarray(kw["radius_body_panda_hand"]).reshape(-1)[0])
            for v in (kw.get(f"radius_body_panda_link{l}"), links.get(str(l)), links.get(l)):
                if v is not None:
                    return float(np.asarray(v).reshape(-1)[0])
            raise MrfError(f"self-collision pair with panda_link{l} needs radius_body_panda_links['{l}']")
        return [radius(a) + radius(b) for a, b in self.self_pairs]

    def set_self_collision_radii(self, rho):
        """Set the pairs' rho on the handle if it changed (one C-ABI call; nothing when the radii are the same)."""
        rho = [float(r) for r in rho]
        if rho != self.self_rho:
            self.fab.set_self_collision([self.self_pairs], [rho])
            self.self_rho = rho

    def compute_action(self, **kwargs) -> np.ndarray:
        rec, obst = self._record_and_obstacles(kwargs)
        if self.self_pairs:
            self.set_self_collision_radii(self._self_collision_radii(kwargs))
        act = self.fab.action_host(rec[None, None, :], obst[None, None] if len(obst) else None, dtype=self.dtype)[0, 0]
        act = np.asarray(act, dtype=np.float64)
        if np.linalg.norm(act) < 1e-6:     # fabrics: "avoid too small actions"
            act = act * 0.0
        return act


def set_planner_panda(degrees_of_freedom: int = 7, nr_obst=0, nr_obst_dyn=1, collision_links_nr=(5,), urdf_links=None,
                      mount_param=None, i_robot=0, device: int = 0, dtype: str = "f64", *, self_collision_pairs=None):
    """Same signature as the reference's set_planner_panda; the URDF constants are compiled into the kernels.
    self_collision_pairs (keyword only): fabrics' dict {"panda_linkN" | "panda_hand": [paired links]}; each pair's rho
    comes from the radius_body_panda_links / radius_body_panda_hand arguments of compute_action."""
    if degrees_of_freedom != 7:
        raise MrfError("the CUDA path is specialised to the 7-dof Panda chain")
    mount = mount_transform(i_robot, mount_param)
    return PandaFabricPlanner(mount, nr_obst, nr_obst_dyn, list(collision_links_nr), i_robot, device, dtype=dtype,
                              self_collision_pairs=self_collision_pairs), PandaGoal()


class PointFabricPlanner:
    """compute_action drop-in for set_planner_point (examples/example_pointmasses_static.py:102-129,
    examples/example_pointmasses_dynamic.py:102-131): 3-dof point robot, mode 'acc'."""

    def __init__(self, n_obstacles: int, n_dyn_obstacles: int = 0, device: int = 0):
        self.n_obst, self.n_dyn = int(n_obstacles), int(n_dyn_obstacles)
        self.fab = Fabrics(config=default_config(1), device=device)

    def _pack(self, kw: dict):
        rec = np.zeros((1, 10))
        rec[0, 0:3] = _vec(kw["q"], 3)
        rec[0, 3:6] = _vec(kw["qdot"], 3)
        rec[0, 6:8] = _vec(kw["x_goal_0"], 2)
        rec[0, 8] = float(np.asarray(kw["weight_goal_0"]).reshape(-1)[0])
        rec[0, 9] = float(np.asarray(kw["radius_body_base_link"]).reshape(-1)[0])
        stat = np.zeros((1, self.n_obst, 4))
        for i in range(self.n_obst):
            x = kw[f"x_obst_{i}"] if f"x_obst_{i}" in kw else kw["x_obsts"][i]
            r = kw[f"radius_obst_{i}"] if f"radius_obst_{i}" in kw else kw["radius_obsts"][i]
            stat[0, i, 0:3] = _vec(x, 3)
            stat[0, i, 3] = float(np.asarray(r).reshape(-1)[0])
        dyn = np.zeros((1, self.n_dyn, 7))
        for i in range(self.n_dyn):
            get = lambda single, plural: kw[f"{single}_{i}"] if f"{single}_{i}" in kw else kw[plural][i]
            dyn[0, i, 0:2] = _vec(get("x_obst_dynamic", "x_obsts_dynamic"))[0:2]
            dyn[0, i, 2:4] = _vec(get("xdot_obst_dynamic", "xdot_obsts_dynamic"))[0:2]
            dyn[0, i, 4:6] = _vec(get("xddot_obst_dynamic", "xddot_obsts_dynamic"))[0:2]
            dyn[0, i, 6] = float(np.asarray(get("radius_obst_dynamic", "radius_obsts_dynamic")).reshape(-1)[0])
        return rec, stat, dyn

    def compute_action(self, **kwargs) -> np.ndarray:
        rec, stat, dyn = self._pack(kwargs)
        act = np.empty((1, 3))
        check(lib().mrf_point_action_host_f64(self.fab.handle.ptr, hptr(rec), self.n_obst, hptr(stat) if self.n_obst else None,
                                              self.n_dyn, hptr(dyn) if self.n_dyn else None, hptr(act), 1),
              "mrf_point_action_host")
        a = act[0]
        if np.linalg.norm(a) < 1e-6:
            a = a * 0.0
        return a


def set_planner_point(goal=None, n_obstacles: int = 2, n_dyn_obstacles: int = 0, device: int = 0):
    """Same role as the reference's set_planner_point (the URDF and the geometry strings are compiled in)."""
    return PointFabricPlanner(n_obstacles, n_dyn_obstacles, device)


# ------------------------------------------------------------------------------------------------------------------
class ForwardFabricsPlanner:
    """Coupled joint-space Rollout Fabrics (forward_planner_Jointspace.py)."""

    def __init__(self, params, planners, N_steps=None, fk_dict=None, goal_struct_robots=None, ROLLOUTS_PLOTTING=0,
                 device: int = 0, dtype: str = "f64", estimate_goal: int = 0):
        self.N_horizon = params.N_HORIZON
        self.dt = params.dt
        self.dof = params.dof
        self.nr_robots = len(self.dof)
        self.nr_obsts = params.nr_obsts
        self.planners = planners
        self.fabrics_mode = params.fabrics_mode
        self.r_robots = params.r_robots
        self.rotation_matrices_pandas = params.rotation_matrix_pandas
        self.collision_links_nrs = params.collision_links_nrs
        self.goal_struct_robots = goal_struct_robots
        self.nr_subgoals = [3] * self.nr_robots
        self.dtype = dtype
        if self.fabrics_mode not in ("vel", "acc"):
            raise MrfError("fabrics_mode must be 'vel' or 'acc'")
        # 'acc' reproduces what the reference's loop does, not a double integrator: the acceleration handed to system_step
        # is reset to zero every step (forward_planner_Jointspace.py:195,202), so q advances with the stored velocity, and
        # the planner's output -- an acceleration in this mode -- is written into q_dot (:233).  The kernels' recurrence
        # (q += dt q_dot; q_dot = action) is exactly that with MrfConfig.mode = 0.
        if len(set(self.nr_obsts)) > 1:
            raise MrfError("the CUDA rollout takes the same number of static spheres for every robot")
        self.radius_obsts = getattr(params, "radius_obsts", None)
        # radius bodies of links > 2 (forward_planner_Jointspace.py:37-40); r_robots[i][z] belongs to link collision_links_nrs[i][z]
        self.r_robots_args = [[self.r_robots[i][z] for z, c in enumerate(self.collision_links_nrs[i]) if c > 2]
                              for i in range(self.nr_robots)]
        r_full = [[0.0] * 8 for _ in range(self.nr_robots)]
        for i in range(self.nr_robots):
            for z, c in enumerate(self.collision_links_nrs[i]):
                if not 1 <= int(c) <= 8:
                    raise MrfError(f"collision link numbers must be 1..8, got {c}")
                r_full[i][int(c) - 1] = float(self.r_robots[i][z])
        mounts = [np.asarray(p.mount) for p in planners]
        cfg = default_config(self.nr_robots, dt=self.dt, static_or_dyn=int(params.STATIC_OR_DYN_FABRICS),
                             mode=1 if self.fabrics_mode == "vel" else 0,
                             mount=mounts, r_robots=r_full, estimate_goal=int(estimate_goal),
                             collision_links=[list(c) for c in self.collision_links_nrs])
        self.fab = Fabrics(config=cfg, device=device)
        # self-collision pairs of the planners the rollouts are built from: rho as the planner last set it, otherwise
        # from this planner's link radii (panda_hand = panda_link8's point and radius)
        pairs, rhos = [], []
        for i, p in enumerate(planners):
            pp = list(getattr(p, "self_pairs", []) or [])
            rho = getattr(p, "self_rho", None)
            if pp and rho is None:
                rad = lambda l, i=i: r_full[i][min(l, 8) - 1]
                rho = [rad(a) + rad(b) for a, b in pp]
                if any(r <= 0.0 for r in rho):
                    raise MrfError(f"robot {i}: a self-collision pair's link has no radius in r_robots; call the planner's "
                                   "compute_action (or set_self_collision_radii) first")
            pairs.append(pp)
            rhos.append(list(rho or []))
        if any(pairs):
            self.fab.set_self_collision(pairs, rhos)

    def forward_multi_fabrics_symbolic(self):
        """The reference builds the CasADi graph here; the CUDA kernels need no per-configuration compilation."""
        return {}

    def _records(self, inputs_action) -> np.ndarray:
        R = self.nr_robots
        rec = np.zeros((1, R, REC))
        for i in range(R):                         # argument order of forward_planner_Jointspace.py:303-329
            rec[0, i, ANG:ANG + 9] = np.asarray(self.rotation_matrices_pandas[i], dtype=np.float64).reshape(9)
            rec[0, i, CON:CON + 4] = _vec(inputs_action["constraints"][i], 4)
            rec[0, i, Q:Q + 7] = _vec(inputs_action["q_robots"][i], 7)
            rec[0, i, QD:QD + 7] = _vec(inputs_action["q_dot_robots"][i], 7)
            rec[0, i, W0] = float(np.asarray(inputs_action["weight_goals0"][i]).reshape(-1)[0])
            rec[0, i, W1] = float(np.asarray(inputs_action["weight_goals1"][i]).reshape(-1)[0])
            rec[0, i, W2] = float(np.asarray(inputs_action["weight_goals2"][i]).reshape(-1)[0])
            rec[0, i, G0:G0 + 3] = _vec(inputs_action["x_goals0"][i], 3)
            rec[0, i, G1:G1 + 3] = _vec(inputs_action["x_goals1"][i], 3)
            rec[0, i, G2] = _vec(inputs_action["x_goals2"][i])[0]
            k = 0
            for l in range(3, 9):                # radius_body_panda_link{l} of the links in the robot's collision set
                if l in self.collision_links_nrs[i]:
                    rec[0, i, RB + l - 3] = float(self.r_robots_args[i][k])
                    k += 1
        return rec

    def _static(self, inputs_action):
        """x_obsts / radius_obsts of the rollout planners (:319-322) -> (1, R, S, 4) or None."""
        S = int(self.nr_obsts[0]) if len(self.nr_obsts) else 0
        if S == 0:
            return None
        if self.radius_obsts is None:
            raise MrfError("params.radius_obsts is needed for rollouts with static obstacles (forward_planner_Jointspace.py:322)")
        st = np.zeros((1, self.nr_robots, S, 4))
        for i in range(self.nr_robots):
            for o in range(S):
                st[0, i, o, 0:3] = _vec(inputs_action["x_obsts"][i][o], 3)
                st[0, i, o, 3] = float(np.asarray(self.radius_obsts[i][o]).reshape(-1)[0])
        return st

    def _rollout(self, inputs_action, trajectories: bool):
        rec, st = self._records(inputs_action), self._static(inputs_action)
        if st is None:
            return self.fab.rollout_host(rec, self.N_horizon, dtype=self.dtype, trajectories=trajectories)
        # static spheres: device entry mrf_rollout_static_dev (tensor hand-off through torch)
        import torch
        from .api import to_soa
        R, N = self.nr_robots, self.N_horizon
        tdt = torch.float64 if self.dtype == "f64" else torch.float32
        dev = f"cuda:{self.fab.device}"
        d_rec = torch.from_numpy(to_soa(rec)).to(dev, dtype=tdt)
        d_st = torch.from_numpy(np.ascontiguousarray(st.transpose(2, 3, 1, 0))).to(dev, dtype=tdt)      # (S,4,R,1)
        t = lambda *shape: torch.empty(shape, dtype=tdt, device=dev)
        avg, xee, gest = t(R, 1), t(R, 3, 1), t(3, 1)
        qN, qdN = (t(R, N, DOF, 1), t(R, N, DOF, 1)) if trajectories else (None, None)
        self.fab.rollout_static_dev(d_rec, d_st, N, avg_vel=avg, x_ee=xee, goal_est=gest, qN=qN, qdN=qdN)
        torch.cuda.synchronize()
        out = {"avg_vel": avg.double().cpu().numpy().T.copy(), "x_ee": xee.double().cpu().numpy().transpose(2, 0, 1).copy(),
               "goal_est": gest.double().cpu().numpy().T.copy()}
        if trajectories:
            out["qN"] = qN.double().cpu().numpy().transpose(3, 0, 1, 2).copy()
            out["qdN"] = qdN.double().cpu().numpy().transpose(3, 0, 1, 2).copy()
        return out

    def get_velocity_rollouts(self, inputs_action):
        """-> list of R arrays of shape (1,): mean square joint velocity over the horizon (:298-336)."""
        out = self._rollout(inputs_action, False)
        self.last = out
        return [np.array([float(out["avg_vel"][0, i])]) for i in range(self.nr_robots)]

    def rollouts_numerical(self, inputs_action=None, **_ignored):
        """-> (q_N, qdot_N, qddot_N) dicts keyed 'robot_i', each [array(7, N)] (:338-423)."""
        out = self._rollout(inputs_action, True)
        self.last = out
        qn, qdn, qddn = {}, {}, {}
        for i in range(self.nr_robots):
            qn[f"robot_{i}"] = [np.asarray(out["qN"][0, i], dtype=np.float64).T.copy()]
            qdn[f"robot_{i}"] = [np.asarray(out["qdN"][0, i], dtype=np.float64).T.copy()]
            qddn[f"robot_{i}"] = [np.zeros((DOF, self.N_horizon))]      # q_ddot is identically 0 in 'vel' mode (:202)
        return qn, qdn, qddn


    def rollouts_numerical_obstacles(self, inputs_action):
        """-> (x, v, a) dicts keyed 'robot_i': per horizon step k an array (3, 8 (R-1)) with the positions / velocities /
        accelerations of the OTHER robots' collision-link spheres as robot i sees them in step k (ascending other robot,
        link1..8) -- the numeric twin of x_obsts_N_fun / v_obsts_N_fun / a_obsts_N_fun
        (forward_planner_Jointspace.py:234-243,283-290,425-511).  Step k evaluates FK at the stepped position q_k with
        the stale velocity qdot_{k-1} (:197-209), v = J qdot, a = Jdot qdot with the reference's sign (utils.py:28);
        STATIC_OR_DYN_FABRICS = 0 zeroes v and a (:215-217)."""
        R, N = self.nr_robots, self.N_horizon
        rec = self._records(inputs_action)
        out = self._rollout(inputs_action, True)
        self.last = out
        q = np.asarray(out["qN"][0], dtype=np.float64)                                  # (R, N, 7): q_k
        qd_prev = np.concatenate([rec[0, :, None, QD:QD + 7], np.asarray(out["qdN"][0], dtype=np.float64)[:, :-1]], axis=1)
        x, v, a = self.fab.kinematics_host(np.ascontiguousarray(q.transpose(1, 0, 2)),
                                           np.ascontiguousarray(qd_prev.transpose(1, 0, 2)))       # (N, R, 8, 3)
        if not self.fab.cfg.static_or_dyn:
            v, a = np.zeros_like(v), np.zeros_like(a)
        xs, vs, as_ = {}, {}, {}
        for i in range(R):
            others = [j for j in range(R) if j != i]
            sel = {j: [int(c) - 1 for c in self.collision_links_nrs[j]] for j in others}                # their collision links
            cat = lambda arr, k: np.concatenate([arr[k, j][sel[j]] for j in others], axis=0).T.copy()   # (3, sum of links)
            xs[f"robot_{i}"] = [cat(x, k) for k in range(N)]
            vs[f"robot_{i}"] = [cat(v, k) for k in range(N)]
            as_[f"robot_{i}"] = [cat(a, k) for k in range(N)]
        return xs, vs, as_


# ------------------------------------------------------------------------------------------------------------------
class _DM:
    """Minimal stand-in for the casadi DM returned by avg_vel_fun (callers use ``.full()[0]``)."""

    def __init__(self, v):
        self._v = np.atleast_2d(np.asarray(v, dtype=np.float64))

    def full(self):
        return self._v


class FabricsRollouts:
    """Decoupled (Cartesian constant-velocity obstacle) rollouts, forward_planner_Cartesian.py."""

    def __init__(self, N, dt, nx, nu, dof, nr_obsts, bool_ring, nr_obsts_dyn=0, v_obsts_dyn=(), fabrics_mode="acc",
                 collision_links_nrs=(7,), nr_constraints=0, radius_sphere=0.08, constraints=None, nr_goals=3,
                 dtype: str = "f64"):
        self.N, self.dt, self.dof = N, dt, dof
        self.Ts, self.nx, self.nu, self.ring = dt, nx, nu, bool_ring
        self.nr_obsts, self.nr_obsts_dyn = nr_obsts, nr_obsts_dyn
        self.v_obsts_dyn = list(v_obsts_dyn)
        self.a_obsts_dyn = [np.zeros((3,))] * len(self.v_obsts_dyn)
        self.fabrics_mode = fabrics_mode
        self.collision_links_nrs = list(collision_links_nrs)
        self.nr_constraints = nr_constraints
        self.radius_sphere = radius_sphere
        self.rotation_matrix_panda = ROT_PANDA.copy()
        self.radius_obsts_dyn, self.radius_obsts = [], []
        self.constraints = constraints
        self.nr_goals = nr_goals
        self.dtype = dtype
        self.radius_body_panda_links = {str(l): np.array(radius_sphere) for l in self.collision_links_nrs if l > 2}
        if fabrics_mode not in ("vel", "acc"):
            raise MrfError("fabrics_mode must be 'vel' or 'acc'")

    # ---- environment-dictionary readers (forward_planner_Cartesian.py:49-69,94-130): host glue, same keys ----
    def preset_radii(self, ob_robot):
        if self.nr_obsts + self.nr_obsts_dyn > 0:
            obst = ob_robot["FullSensor"]["obstacles"]
            first = list(obst.keys())[0]
            self.radius_obsts = [obst[first + i]["size"] for i in range(self.nr_obsts)]
            self.radius_obsts_dyn = [obst[first + self.nr_obsts + i]["size"] for i in range(self.nr_obsts_dyn)]
        else:
            self.radius_obsts_dyn, self.radius_obsts = [], []

    def get_x_obsts(self, ob_robot) -> list:
        obst = ob_robot["FullSensor"]["obstacles"]
        first = list(obst.keys())[0]
        return [obst[first + i]["position"] for i in range(self.nr_obsts)]

    def get_x_obsts_dyn_current(self, ob_robot) -> list:
        obst = ob_robot["FullSensor"]["obstacles"]
        first = list(obst.keys())[0]
        return [obst[first + self.nr_obsts + i]["position"] for i in range(self.nr_obsts_dyn)]

    def get_goal_x_weight(self, ob_robot, goal):
        goals = ob_robot["FullSensor"]["goals"]
        first = list(goals.keys())[0]
        x_goals = [goals[first + i]["position"] for i in range(self.nr_goals)]
        weight_goals = [goal.sub_goals()[i].weight() for i in range(self.nr_goals)]
        return x_goals, weight_goals

    def preset_radii_obsts_dyn(self, radii_obst_dyn):
        self.radius_obsts_dyn = radii_obst_dyn

    def system_step(self, pos, vel, input, dt: float, fabrics_mode="vel"):  # noqa: A002 (the reference's argument name)
        """forward_planner_Cartesian.py:77-92."""
        pos = np.asarray(pos, dtype=np.float64)
        inp = np.asarray(input, dtype=np.float64)
        if fabrics_mode == "acc":
            vel = np.asarray(vel, dtype=np.float64)
            return pos + dt * vel + 0.5 * dt ** 2 * inp, vel + dt * inp
        if fabrics_mode == "vel":
            return pos + dt * inp, inp
        print("nonexisting fabrics mode inserted, should be vel or acc")
        return [], []

    def get_action(self, planner, pos, vel, x_obsts: list, x_obsts_dyn: list, x_goals: list, weight_goals: list):
        """One planner.compute_action with this rollout object's constants (forward_planner_Cartesian.py:132-191)."""
        x_goals, weight_goals = list(x_goals), list(weight_goals)
        for _ in range(3 - self.nr_goals):              # "append some zeros" (:145-149)
            x_goals.append(0)
            weight_goals.append(0)
        return planner.compute_action(
            q=pos, qdot=vel, angle_goal_1=self.rotation_matrix_panda, x_goal_0=x_goals[0], x_goal_1=x_goals[1],
            x_goal_2=x_goals[2], weight_goal_0=weight_goals[0], weight_goal_1=weight_goals[1], weight_goal_2=weight_goals[2],
            x_obsts=x_obsts, radius_obsts=self.radius_obsts, x_obsts_dynamic=x_obsts_dyn, xdot_obsts_dynamic=self.v_obsts_dyn,
            xddot_obsts_dynamic=[np.array([0.0, 0.0, 0.0])] * self.nr_obsts_dyn, radius_obsts_dynamic=self.radius_obsts_dyn,
            radius_body_panda_links=self.radius_body_panda_links, radius_body_panda_hand=np.array([0.08]),
            constraint_0=self.constraints)

    def get_x_obsts_dyn_N(self, x_obsts_dyn):
        """Constant-velocity obstacle positions along the horizon, both forms of forward_planner_Cartesian.py:195-216:
        a list of N+1 arrays (3, nr_obsts_dyn) (k = 0..N) and a list of N lists of per-obstacle positions (k = 0..N-1)."""
        x0 = np.stack(x_obsts_dyn).transpose()
        v = np.stack(self.v_obsts_dyn).transpose()
        x_N = [x0]
        for _ in range(self.N):
            x_N.append(x_N[-1] + v * self.dt)
        x_list = [[[] for _ in range(self.nr_obsts_dyn)] for _ in range(self.N)]
        x_list[0] = np.array(x_obsts_dyn)
        for i in range(self.N - 1):
            for o in range(self.nr_obsts_dyn):
                x_list[i + 1][o] = x_list[i][o] + self.v_obsts_dyn[o] * self.dt
        return x_N, x_list

    def forward_fabrics(self, planner, pos_k, vel_k, ob_robot, goal, x_obsts_dyn_0=None, x_goals_struct=None,
                        weight_goals_struct=None):
        """"The Python rollout loop" (forward_planner_Cartesian.py:218-273): N x (compute_action, system_step) with the
        obstacles at x0 + k dt v.  Every action comes from the CUDA action kernel through planner.compute_action.
        -> (q_stacked, qdot_stacked, qddot_stacked) lists over the horizon."""
        u_k = []
        q_stacked, qdot_stacked, qddot_stacked = [], [], []
        for i in range(self.N):
            x_obsts = self.get_x_obsts(ob_robot) if self.nr_obsts > 0 else []
            if self.nr_obsts_dyn > 0:
                x_dyn = self.get_x_obsts_dyn_current(ob_robot) if x_obsts_dyn_0 is None else x_obsts_dyn_0
                _, x_dyn_list = self.get_x_obsts_dyn_N(x_dyn)
            else:
                x_dyn_list = [[] for _ in range(self.N)]
            if x_goals_struct is None:
                x_goals, weight_goals = self.get_goal_x_weight(ob_robot, goal)
            else:
                x_goals, weight_goals = list(x_goals_struct.values()), list(weight_goals_struct.values())
            u_k[0:self.dof] = self.get_action(planner, pos_k, vel_k, x_obsts=x_obsts, x_obsts_dyn=x_dyn_list[i],
                                              x_goals=x_goals, weight_goals=weight_goals)
            pos_k, vel_k = self.system_step(pos_k, vel_k, u_k[0:self.dof], dt=self.dt, fabrics_mode=self.fabrics_mode)
            if self.fabrics_mode == "acc":
                qddot_stacked.append(u_k.copy())
                qdot_stacked.append(vel_k.copy())
            else:
                qdot_stacked.append(u_k.copy())
            q_stacked.append(pos_k.copy())
        return q_stacked, qdot_stacked, qddot_stacked

    def x_obsts_dyn_numerical(self, pos_obsts_dyn):
        """-> list over k = 0..N-1 of arrays (3, nr_obsts_dyn): obstacle positions AFTER step k
        (x_obsts_dyn_N_fun, forward_planner_Cartesian.py:448-458,471-474,491-505)."""
        x = np.stack([np.asarray(p, dtype=np.float64).reshape(3) for p in pos_obsts_dyn])
        v = np.stack([np.asarray(p, dtype=np.float64).reshape(3) for p in self.v_obsts_dyn])
        out = []
        for _ in range(self.N):
            x = x + self.dt * v
            out.append(x.T.copy())
        return out

    def reset_v_obsts_dyn(self, v_obsts_dyn):
        self.v_obsts_dyn = v_obsts_dyn

    def symbolic_forward_fabrics(self, planner, goal_struct):
        self.planner = planner
        self.nr_subgoals = len(goal_struct._config)
        if (planner.fab.cfg.mode == 1) != (self.fabrics_mode == "vel"):
            raise MrfError("the planner was concretized in a different mode than fabrics_mode of the rollouts")
        return {}

    def define_arguments_numerical(self, q_robot, q_dot_robot, weight_goals, x_goals, x_obsts, x_obsts_dyn, v_obsts_dyn,
                                   constraints=()):
        """Same flat argument list as forward_planner_Cartesian.py:507-536."""
        a = []
        if self.nr_subgoals > 1:
            a.append(self.rotation_matrix_panda)
        for _ in range(self.nr_constraints):
            a.append(constraints)
        a.append(q_robot)
        a.append(q_dot_robot)
        for i in range(self.nr_subgoals):
            a.append(weight_goals["subgoal" + str(i)])
        for i in range(self.nr_subgoals):
            a.append(x_goals["subgoal" + str(i)])
        for i in range(self.nr_obsts):
            a.append(x_obsts[i])
        for i in range(self.nr_obsts):
            a.append(self.radius_obsts[i])
        if self.nr_obsts + self.nr_obsts_dyn > 0:
            for r in self.radius_body_panda_links.values():
                a.append(r)
        for r in self.radius_obsts_dyn:
            a.append(r)
        for i in range(self.nr_obsts_dyn):
            a.append(x_obsts_dyn[i])
        for i in range(self.nr_obsts_dyn):
            a.append(v_obsts_dyn[i])
        for i in range(self.nr_obsts_dyn):
            a.append(self.a_obsts_dyn[i] if i < len(self.a_obsts_dyn) else np.zeros(3))
        self.arguments = a
        return a

    def _unpack(self, arguments):
        it = iter(arguments)
        rec = np.zeros(REC)
        if self.nr_subgoals > 1:
            rec[ANG:ANG + 9] = np.asarray(next(it), dtype=np.float64).reshape(9)
        for _ in range(self.nr_constraints):
            rec[CON:CON + 4] = _vec(next(it), 4)
        rec[Q:Q + 7] = _vec(next(it), 7)
        rec[QD:QD + 7] = _vec(next(it), 7)
        w = [float(np.asarray(next(it)).reshape(-1)[0]) for _ in range(self.nr_subgoals)]
        g = [_vec(next(it)) for _ in range(self.nr_subgoals)]
        rec[W0], rec[G0:G0 + 3] = w[0], g[0]
        if self.nr_subgoals > 1:
            rec[W1], rec[G1:G1 + 3] = w[1], g[1]
        if self.nr_subgoals > 2:
            rec[W2], rec[G2] = w[2], g[2][0]
        xs = [_vec(next(it), 3) for _ in range(self.nr_obsts)]
        rs = [float(np.asarray(next(it)).reshape(-1)[0]) for _ in range(self.nr_obsts)]
        if self.nr_obsts + self.nr_obsts_dyn > 0:
            for i, l in enumerate(range(3, 9)):
                if str(l) in self.radius_body_panda_links:
                    rec[RB + i] = float(np.asarray(next(it)).reshape(-1)[0])
        rd = [float(np.asarray(next(it)).reshape(-1)[0]) for _ in range(len(self.radius_obsts_dyn))]
        xd = [_vec(next(it), 3) for _ in range(self.nr_obsts_dyn)]
        vd = [_vec(next(it), 3) for _ in range(self.nr_obsts_dyn)]
        obst = np.zeros((self.nr_obsts + self.nr_obsts_dyn, OBST))
        for i in range(self.nr_obsts):
            obst[i, 0:3], obst[i, 9] = xs[i], rs[i]
        for i in range(self.nr_obsts_dyn):
            o = self.nr_obsts + i
            obst[o, 0:3], obst[o, 3:6], obst[o, 9] = xd[i], vd[i], rd[i]
        return rec, obst

    def _run(self, arguments):
        rec, obst = self._unpack(arguments)
        return self.planner.fab.rollout_cart_host(0, rec[None], obst[None], self.N, dtype=self.dtype)

    def rollouts_numerical(self, arguments):
        """-> q_N, qdot_N, qddot_N, each array (7, N) (forward_planner_Cartesian.py:538-559).  'vel' mode: q_ddot is
        identically 0 (:431-433); 'acc' mode: the actions, recovered from the velocity steps (vel += dt * action, :84)."""
        rec, _ = self._unpack(arguments)
        _, qN, qdN = self._run(arguments)
        q = np.asarray(qN[0], dtype=np.float64).T.copy()
        qd = np.asarray(qdN[0], dtype=np.float64).T.copy()
        if self.fabrics_mode == "vel":
            return q, qd, np.zeros((DOF, self.N))
        prev = np.concatenate([rec[QD:QD + 7, None], qd[:, :-1]], axis=1)
        return q, qd, (qd - prev) / self.dt

    def get_velocity_rollouts(self, arguments):
        avg, _, _ = self._run(arguments)
        return _DM([float(avg[0])])


# ------------------------------------------------------------------------------------------------------------------
class deadlockprevention:  # noqa: N801 (the reference's class name)
    """deadlock_prevention.py drop-in; the check itself runs in the CUDA deadlock kernel (B = 1)."""

    def __init__(self, dof, n_robots, N_horizon, device: int = 0):
        self.dof, self.n_robots, self.N_horizon = dof, n_robots, N_horizon
        if dof[0] == 2:      # point-mass constants (deadlock_prevention.py:12-19)
            kw = dict(dl_avg_vel_constant=0.03, dl_dist_constant=1.0, dl_goal_weight_follower=10.0, dl_goal_weight_leader=1.0,
                      dl_time_wait=50, dl_nr_goal_scale=100.0)
        else:                # manipulators (:20-27) = the library defaults
            kw = {}
        self.avg_vel_constant = kw.get("dl_avg_vel_constant", 0.16)
        self.dist_constant = kw.get("dl_dist_constant", 0)
        self.goal_weight_follower = int(kw.get("dl_goal_weight_follower", 2))
        self.goal_weight_leader = int(kw.get("dl_goal_weight_leader", 3))
        self.time_wait = kw.get("dl_time_wait", 300)
        self.nr_goal_scale = int(kw.get("dl_nr_goal_scale", 2))
        self.fab = Fabrics(config=default_config(n_robots, **kw), device=device)
        self._st_int = np.array([[0, 1, 0, 1]], dtype=np.int32)      # i_leader, i_follower, i_robots_dead (:10-11,33)
        self._st_goal = np.zeros((1, 3))
        self.deadlock = False

    @property
    def i_leader(self):
        return int(self._st_int[0, 0])

    @property
    def i_follower(self):
        return int(self._st_int[0, 1])

    @property
    def goal_robot0(self):
        return self._st_goal[0].copy()

    def compute_velocity_average(self, q_dot_robots_N):
        """deadlock_prevention.py:36-43 (mean ABSOLUTE joint velocity; unused by the examples, host arithmetic)."""
        avg_sum = 0
        for i in range(self.n_robots):
            for df in range(self.dof[i]):
                q = np.abs(np.asarray(q_dot_robots_N["robot_" + str(i)][df], dtype=np.float64))
                avg_sum = avg_sum + q.sum() / (self.N_horizon * self.dof[i])
        return avg_sum

    def compute_distance_to_goal(self, x_robot, goal_robot):
        return np.linalg.norm(np.asarray(x_robot) - np.asarray(goal_robot))

    def deadlock_checking(self, x_robots, goal_robots, goal_weights, time_step, time_deadlock_out, avg_sum,
                          state_machine_robots=()):
        R = self.n_robots
        dim = int(np.asarray(x_robots[0]).size)
        if dim == 2:       # planar point robots: pad z = 0 (norms unchanged bit for bit) and strip it again below
            pad = lambda seq: [np.append(np.asarray(v, dtype=np.float64).reshape(2), 0.0) for v in seq]
            g3 = pad(goal_robots)
            out_g, out_w, tdo = self.deadlock_checking(pad(x_robots), g3, goal_weights, time_step, time_deadlock_out, avg_sum,
                                                       state_machine_robots)
            if self.deadlock:
                # the reference reads goal_robot0[2] (deadlock_prevention.py:99) -- an IndexError for 2-D positions
                raise IndexError("index 2 is out of bounds for axis 0 with size 2")
            for i in range(R):
                if out_g[i][:2].tolist() != np.asarray(goal_robots[i], dtype=np.float64).reshape(2).tolist():
                    goal_robots[i] = out_g[i][:2].copy()
            return goal_robots, out_w, tdo
        # the reference indexes state_machine_robots[z[0]] for every pair (deadlock_prevention.py:62): a short list is an
        # IndexError there, and would be an out-of-bounds read in the kernel
        if len(state_machine_robots) != R or len(x_robots) != R or len(goal_robots) != R or len(goal_weights) != R:
            raise IndexError(f"deadlock_checking: x_robots, goal_robots, goal_weights and state_machine_robots need one "
                             f"entry per robot ({R})")
        x = np.ascontiguousarray(np.stack([_vec(v, 3) for v in x_robots])[None])
        g = np.ascontiguousarray(np.stack([_vec(v, 3) for v in goal_robots])[None])
        w = np.ascontiguousarray(np.array([[float(np.asarray(v).reshape(-1)[0]) for v in goal_weights]]))
        a = np.array([float(np.asarray(avg_sum).reshape(-1)[0])])
        sm = np.ascontiguousarray(np.array([list(state_machine_robots)], dtype=np.int32))
        ts = np.array([int(time_step)], dtype=np.int32)
        tdo = np.array([int(time_deadlock_out)], dtype=np.int32)
        flag = np.zeros(1, dtype=np.int32)
        check(lib().mrf_deadlock_host_f64(self.fab.handle.ptr, hptr(x), hptr(g), hptr(w), hptr(a), hptr(sm), hptr(ts),
                                          hptr(tdo), hptr(self._st_int), hptr(self._st_goal), hptr(flag), 1),
              "mrf_deadlock_host")
        self.deadlock = bool(flag[0])
        # the reference mutates the caller's lists in place (this is how the follower goal reaches compute_action)
        for i in range(R):
            if g[0, i].tolist() != _vec(goal_robots[i], 3).tolist():
                goal_robots[i] = g[0, i].copy()
            if w[0, i] != float(np.asarray(goal_weights[i]).reshape(-1)[0]):
                goal_weights[i] = w[0, i]
        return goal_robots, goal_weights, int(tdo[0])


# ------------------------------------------------------------------------------------------------------------------
class StateMachine:
    """state_machine.py drop-in (Panda branch): the decision logic runs in the CUDA fsm kernel with B = 1.
    `fk_fun_ee(q)` may be any callable returning the hand position (the reference passes a CasADi function)."""

    def __init__(self, start_goal, nr_robots, nr_blocks, fk_fun_ee, robot_types, device: int = 0):
        import torch
        self.torch = torch
        self.fk_fun_ee = fk_fun_ee
        self.nr_blocks_panda = nr_blocks
        self.start_goal = np.asarray(start_goal, dtype=np.float64).reshape(3)
        self.fab = Fabrics(config=default_config(1), device=device)
        dev = f"cuda:{device}"
        t = lambda a, dt=torch.float64: torch.tensor(a, dtype=dt, device=dev)
        self._start = t(self.start_goal).reshape(1, 3, 1)
        self._goal = self._start.clone()
        self._above = torch.zeros((1, 3, 1), dtype=torch.float64, device=dev)
        self._weight = t([[2.0]])
        self._st = t([[[1]], [[0]], [[0]], [[0]], [[0]], [[0]]], torch.int32)
        self._grip = torch.zeros((1, 2, 1), dtype=torch.float64, device=dev)
        self._dev = dev

    def get_state_machine_panda(self, q_robot, q_robot_gripper, goal_block, robot_type="panda"):
        t = self.torch
        x = np.asarray(self.fk_fun_ee(q_robot), dtype=np.float64).reshape(3)
        mk = lambda a, n: t.tensor(np.asarray(a, dtype=np.float64).reshape(1, n, 1), dtype=t.float64, device=self._dev)
        self.fab.fsm_dev([int(self.nr_blocks_panda)], mk(x, 3), mk(q_robot_gripper, 2), mk(goal_block, 3), self._start,
                         self._goal, self._above, self._weight, self._st, self._grip)
        t.cuda.synchronize()
        return int(self._st[0, 0, 0])

    @property
    def state_machine_panda(self):
        return int(self._st[0, 0, 0])

    def get_goal_robot(self):
        return self._goal[0, :, 0].cpu().numpy()

    def get_weight_goal0(self):
        w = float(self._weight[0, 0])
        return int(w) if w == int(w) else w

    def get_nr_blocks_picked(self):
        return int(self._st[1, 0, 0])

    def get_success_rate(self):
        return (int(self._st[1, 0, 0]) - int(self._st[2, 0, 0])) / self.nr_blocks_panda

    # small read-outs of the reference class (state_machine.py:50-67,130-131); host side, the hand position comes from
    # the same `fk_fun_ee` callable the decision step uses
    def get_x_ee(self, q_robot):
        return np.asarray(self.fk_fun_ee(q_robot), dtype=np.float64).reshape(3)

    def get_distance_ee_goal(self, q_robot, goal):
        return float(np.linalg.norm(self.get_x_ee(q_robot)[:2] - np.asarray(goal, dtype=np.float64).reshape(-1)[:2]))

    def get_distance_ee_goal3(self, q_robot, goal):
        return float(np.linalg.norm(self.get_x_ee(q_robot) - np.asarray(goal, dtype=np.float64).reshape(3)))

    def get_distance_ee_start(self, q_robot):
        return float(np.linalg.norm(self.get_x_ee(q_robot) - self.start_goal))

    def get_gripper_status(self):
        return ("close" if int(self._st[4, 0, 0]) else "open"), "open"   # (panda, second-robot slot: unused for Pandas)

    def get_gripper_action_panda(self, q_panda_gripper):
        """The action computed with the last get_state_machine_panda call's gripper state (same q as the reference's
        call order, example_pandas_Jointspace.py:301,447)."""
        q = np.asarray(q_panda_gripper, dtype=np.float64).reshape(2)
        closed = int(self._st[4, 0, 0])
        a = np.zeros(2)
        if closed:
            a[:] = -0.05
        elif np.linalg.norm(q - np.array([0.04, 0.04])) > 0.005:
            a = np.where(q > 0.04, -0.4, 0.4)
        return a
