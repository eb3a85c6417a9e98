"""Closed-loop batched episodes: the control loop of examples/example_pandas_Jointspace.py:280-458 for thousands of
independent scenarios at once, entirely on the GPU (SURVEY.md 8f rank 2; no pybullet).

Per control step, for every scenario (file:line in examples/example_pandas_Jointspace.py):
  1. end-effector FK and the RF-CV goal estimate of robot 1                :324-348   (rollout kernel pre-pass)
  2. coupled Rollout-Fabrics horizon -> mean-square velocity per robot     :352-376   (rollout kernel, weight_goal_1 = 10)
  3. deadlock_checking -> follower goal / weights / timer                   :379-385   (deadlock kernel)
  4. other robots' collision spheres (n_obst_per_link, link-origin velocity):400-412   (obstacles kernel)
  5. executed action per robot (weight_goal_1 = 20), velocity clip          :417-453   (action kernel)
  6. kinematic environment step q += dt * clip(action)  (urdfenvs 'vel' mode stand-in for pybullet, :454)
Two task protocols.  Reach task (default): every robot keeps its goal, state-machine code 0 ("move to goal"), and an
episode succeeds when every hand is within `epsilon` (0.05, the goal struct's epsilon, :35) of its own goal.
Pick-and-place (`blocks=`, `start_goal=`): the reference's state machine (others_planner/state_machine.py) runs on the
device every step -- it sets goals / weight_goal_0, gates the deadlock logic, switches to the obstacle-free grasp
planner in state 2, holds the arm while gripping / releasing and drives the finger joints; blocks are kinematic (picked
in order, never dropped); an episode succeeds when every robot has picked all its blocks (state 10).  One control step is ONE C-ABI call (mrf_episode_step_dev_*: seven kernel launches), captured in a CUDA
graph and replayed; torch only owns the tensors.

Two rollout models (`rollouts=`).  "jointspace" (default) is the loop above: coupled ForwardFabricsPlanner rollouts.
"cartesian" is the loop of examples/example_pandas_cartesian.py:295-462 (decoupled FabricsRollouts, one per robot):
  1. velocity clip; end-effector FK and J qdot at the measured state; RF-CV goal of robot 1 = x_ee + 0.2 * J qdot
     (the true hand velocity, estimate_goal = 2), written into its goal before the rollouts      :343-357
  2. other robots' collision spheres with their true sphere velocities (compute_x_obsts_dyn_0)   :343-352
  3. each robot's Cartesian rollout against those spheres moving at constant velocity, weight_goal_1 = 20 in the
     rollouts as in the action (:42); all robots in one launch                                  :361-418
  4. deadlock_checking on sum(avg_vel) / R                                                      :405
  5.-6. obstacle staging with link-origin velocities, executed action, integration: as in the joint-space loop
     (the Cartesian example's action-side staging is taken to be the joint-space example's).
The rollouts always use the planner with collision links (no grasp planner inside the horizon), as the coupled ones do.

BatchedPointEpisodes runs the loops of the two point-mass examples (examples/example_pointmasses_static.py, _dynamic.py):
many control steps per kernel launch, see its docstring.
"""
from __future__ import annotations

import numpy as np

from ._lib import G0, Q, QD, W0, W1, MrfError
from .api import Fabrics, to_soa

VEL_LIMITS = [2.175, 2.175, 2.175, 2.175, 2.61, 2.61, 2.61]          # example_pandas_Jointspace.py:221
ROLLOUT_MODELS = {"jointspace": 0, "cartesian": 1}                    # MrfEpisode.rollout_model


class BatchedEpisodes:
    def __init__(self, rec: np.ndarray, n_horizon: int = 10, rollout_fabrics: bool = True, resolve_deadlocks: bool = True,
                 estimate_goal: bool = False, static_or_dyn: int = 1, n_obst_per_link: int = 1, device: int = 0,
                 dtype: str = "f32", epsilon: float = 0.05, use_graph: bool = True, blocks=None, start_goal=None,
                 rollouts: str = "jointspace"):
        import torch
        self.torch = torch
        if rollouts not in ROLLOUT_MODELS:
            raise MrfError(f"rollouts must be one of {sorted(ROLLOUT_MODELS)}, got {rollouts!r}")
        if rollouts == "cartesian" and not rollout_fabrics:
            raise MrfError('rollouts="cartesian" needs rollout_fabrics=True (MRDF runs no rollouts)')
        self.rollout_model = ROLLOUT_MODELS[rollouts]
        B, R, _ = rec.shape
        self.B, self.R, self.N = B, R, int(n_horizon)
        self.rollout_fabrics, self.resolve_deadlocks = rollout_fabrics, resolve_deadlocks
        self.n_per_link, self.epsilon, self.use_graph = int(n_obst_per_link), float(epsilon), use_graph
        self.dev = torch.device(f"cuda:{device}")
        self.tdt = torch.float32 if dtype == "f32" else torch.float64
        # RF-CV goal estimate: Jacobian column 0 in the joint-space example (:346-348), J qdot in the Cartesian one (:355-357)
        est_mode = (2 if self.rollout_model == 1 else 1) if estimate_goal else 0
        self.fab = Fabrics(R, device=device, estimate_goal=est_mode, static_or_dyn=static_or_dyn)
        self.fab.handle.set_coop_max_batch(0 if B > 256 else 1 << 20)
        t = lambda a, dt=None: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev, dtype=dt or self.tdt)
        self.rec = t(to_soa(rec))                                    # (44,R,B): q, qdot rows are the live state
        self.goal0 = self.rec[G0:G0 + 3].permute(1, 0, 2).contiguous().clone()     # (R,3,B) task goals
        self.w0 = self.rec[W0].clone()                                              # (R,B)
        z = lambda *s, dt=None: torch.zeros(s, dtype=dt or self.tdt, device=self.dev)
        self.avg, self.xee, self.gest = z(R, B), z(R, 3, B), z(3, B)
        self.obst = z(8 * self.n_per_link * (R - 1), 10, R, B)
        self.act = z(7, R, B)
        self.sm = z(R, B, dt=torch.int32)                                            # state-machine code 0
        self.tstep = z(B, dt=torch.int32)
        self.tdo = torch.full((B,), 1000, dtype=torch.int32, device=self.dev)       # :275
        self.st_int = torch.tensor([0, 1, 0, 1], dtype=torch.int32, device=self.dev).repeat_interleave(B).contiguous()
        self.st_goal = z(3, B)
        self.flag = z(B, dt=torch.int32)
        self.dt = float(self.fab.cfg.dt)
        # metrics
        self.done_at = torch.full((B,), -1, dtype=torch.int32, device=self.dev)
        self.deadlock_steps = z(B, dt=torch.int32)
        self.nonfinite_steps = z(B, dt=torch.int32)     # control steps with a non-finite executed action (arm held still)
        self.min_clear = torch.full((B,), 100.0, dtype=self.tdt, device=self.dev)   # :231 min_clearance = 100
        self.sx = z(8 * self.n_per_link, 3, R, B)
        # pick-and-place task: blocks (B, n_blocks, R, 3) rest positions, start_goal (B, R, 3)
        self.pick_and_place = blocks is not None
        if self.pick_and_place:
            blocks = np.asarray(blocks, dtype=np.float64)
            self.n_blocks = blocks.shape[1]
            self.blocks = t(np.transpose(blocks, (1, 2, 3, 0)))                      # (n_blocks,R,3,B)
            self.start_goal = t(np.transpose(np.asarray(start_goal, dtype=np.float64), (1, 2, 0)))   # (R,3,B)
            self.q_grip = torch.full((R, 2, B), 0.04, dtype=self.tdt, device=self.dev)
            self.goal_block, self.fsm_above, self.grip_action = z(R, 3, B), z(R, 3, B), z(R, 2, B)
            self.fsm_st = z(6, R, B, dt=torch.int32)
            self.fsm_st[0].fill_(1)                                                   # state_machine.py:8
            self.goal0.copy_(self.start_goal)                                         # :33
            self.w0.fill_(2.0)                                                        # :34
            self.kin_scratch = z(3, 8, 3, R, B)
        if self.rollout_model == 1 and not self.pick_and_place:
            self.kin_scratch = z(3, 8, 3, R, B)                                       # hand FK and J qdot
        self.graph = None
        self.steps_done = 0
        self._ep = None

    def _episode_struct(self):
        """The MrfEpisode argument of mrf_episode_step_dev_* (built once: the tensors never move)."""
        import ctypes as C
        from ._lib import MrfEpisode
        from .spheres import sphere_offsets
        R, B = self.R, self.B
        self._offsets = np.ascontiguousarray(sphere_offsets(self.n_per_link), dtype=np.float64)
        if not self.rollout_fabrics and not self.pick_and_place:
            self.kin_scratch = self.torch.zeros((3, 8, 3, R, B), dtype=self.tdt, device=self.dev)
        ep = MrfEpisode()
        ep.struct_size = C.sizeof(MrfEpisode)
        ep.n_horizon, ep.rollout_fabrics, ep.resolve_deadlocks = self.N, int(self.rollout_fabrics), int(self.resolve_deadlocks)
        ep.rollout_model = self.rollout_model
        w1_rollout = 20.0 if self.rollout_model == 1 else 10.0          # example_pandas_cartesian.py:42 / _Jointspace.py:43
        ep.n_per_link, ep.epsilon, ep.w1_rollout, ep.w1_action, ep.clearance_radius_sum = self.n_per_link, self.epsilon, w1_rollout, 20.0, 0.16
        for i, v in enumerate(VEL_LIMITS):
            ep.vel_limit[i] = v
        ep.offsets = self._offsets.ctypes.data
        p = lambda t: None if t is None else t.data_ptr()
        ep.rec, ep.goal0, ep.w0, ep.avg_vel, ep.x_ee, ep.goal_est = p(self.rec), p(self.goal0), p(self.w0), p(self.avg), p(self.xee), p(self.gest)
        ep.obst, ep.spheres_x, ep.action = p(self.obst), p(self.sx), p(self.act)
        ep.kin_scratch = p(getattr(self, "kin_scratch", None))
        ep.sm_state, ep.time_step, ep.time_deadlock_out, ep.st_int, ep.st_goal = p(self.sm), p(self.tstep), p(self.tdo), p(self.st_int), p(self.st_goal)
        ep.flag, ep.done_at, ep.deadlock_steps, ep.min_clearance = p(self.flag), p(self.done_at), p(self.deadlock_steps), p(self.min_clear)
        ep.nonfinite_steps = p(self.nonfinite_steps)
        if self.pick_and_place:
            ep.pick_and_place, ep.n_blocks = 1, self.n_blocks
            ep.blocks, ep.start_goal, ep.q_grip, ep.goal_block = p(self.blocks), p(self.start_goal), p(self.q_grip), p(self.goal_block)
            ep.fsm_above, ep.fsm_st, ep.grip_action = p(self.fsm_above), p(self.fsm_st), p(self.grip_action)
        return ep

    # one control step = one C-ABI call = seven kernel launches on the current stream (graph-capturable)
    def _step(self):
        import ctypes as C
        from ._lib import check, lib
        if self._ep is None:
            self._ep = self._episode_struct()
        fn = lib().mrf_episode_step_dev_f32 if self.tdt == self.torch.float32 else lib().mrf_episode_step_dev_f64
        check(fn(self.fab.handle.ptr, C.byref(self._ep), self.B, self.torch.cuda.current_stream(self.dev).cuda_stream),
              "mrf_episode_step_dev")

    def run(self, n_steps: int):
        torch = self.torch
        if self.use_graph and self.graph is None:
            s = torch.cuda.Stream(device=self.dev)
            s.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(s):
                for _ in range(2):                      # warm-up outside the capture
                    self._step()
            torch.cuda.current_stream(self.dev).wait_stream(s)
            self.steps_done += 2
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):          # capture records the launches, it does not execute them
                self._step()
            n_steps -= 2
        for _ in range(max(0, n_steps)):
            if self.graph is not None:
                self.graph.replay()
            else:
                self._step()
            self.steps_done += 1
        return self

    def results(self) -> dict:
        self.torch.cuda.synchronize(self.dev)
        done = self.done_at.cpu().numpy()
        extra = {}
        if self.pick_and_place:
            extra = {"state": self.fsm_st[0].T.cpu().numpy(), "blocks_picked": self.fsm_st[1].T.cpu().numpy(),
                     "q_grip": self.q_grip.permute(2, 0, 1).double().cpu().numpy()}
        return {**extra, "steps": self.steps_done, "success": done >= 0, "steps_to_success": done,
                "deadlock_steps": self.deadlock_steps.cpu().numpy(),
                "nonfinite_steps": self.nonfinite_steps.cpu().numpy(),
                "min_clearance": self.min_clear.double().cpu().numpy(),
                "q": self.rec[Q:Q + 7].permute(2, 1, 0).double().cpu().numpy(),
                "x_ee": (self.xee.permute(2, 0, 1) if (self.rollout_fabrics or self.pick_and_place) else
                         self.kin_scratch[0, 7].permute(2, 1, 0)).double().cpu().numpy()}


class BatchedPointEpisodes:
    """Closed-loop point-mass episodes: the control loops of examples/example_pointmasses_static.py (dynamic=False) and
    examples/example_pointmasses_dynamic.py (dynamic=True) for B independent scenarios of R = 2..8 point robots (3 dof:
    x, y, theta), entirely on the GPU.  Every call of run(n) is ONE C-ABI call, mrf_point_episode_run_dev_*, that runs n
    control steps in one kernel launch with the state in registers; the loop itself (obstacles, planner, integration,
    metrics) is documented at MrfPointEpisode in include/mrf_b200.h.  Splitting an episode over several run() calls
    gives the same bits as one call.

      q0 (B,R,3), goals (B,R,2), scene (B,S,4) x, y, z, radius of S <= 16 scene spheres (or None), radius / weight:
      body radius and weight_goal_0 (scalars or (B,R)), qdot0 (B,R,3) (default 0).
    An episode succeeds when every robot is within `epsilon` of its goal in (x, y).  The reference's point examples do
    not record a goal tolerance; the default 0.05 is the Panda loop's (BatchedEpisodes).  dt and the planner constants
    come from default_config(1), the handle PointFabricPlanner uses.
    """

    def __init__(self, q0, goals, scene=None, dynamic: bool = False, radius=0.2, weight=1.0, qdot0=None,
                 epsilon: float = 0.05, dtype: str = "f32", device: int = 0, record: bool = False):
        import torch
        from ._lib import default_config
        self.torch = torch
        q0 = np.asarray(q0, dtype=np.float64)
        if q0.ndim != 3 or q0.shape[2] != 3:
            raise MrfError(f"q0 must be (B, R, 3), got {q0.shape}")
        B, R, _ = q0.shape
        goals = np.asarray(goals, dtype=np.float64)
        if goals.shape != (B, R, 2):
            raise MrfError(f"goals must be ({B}, {R}, 2), got {goals.shape}")
        scene = np.zeros((B, 0, 4)) if scene is None else np.asarray(scene, dtype=np.float64)
        if scene.ndim != 3 or scene.shape[0] != B or scene.shape[2] != 4:
            raise MrfError(f"scene must be ({B}, S, 4), got {scene.shape}")
        qdot0 = np.zeros((B, R, 3)) if qdot0 is None else np.asarray(qdot0, dtype=np.float64)
        if qdot0.shape != (B, R, 3):
            raise MrfError(f"qdot0 must be ({B}, {R}, 3), got {qdot0.shape}")
        if dtype not in ("f32", "f64"):
            raise MrfError(f"dtype must be 'f32' or 'f64', got {dtype!r}")
        self.B, self.R, self.S = B, R, scene.shape[1]
        self.dynamic, self.epsilon, self.record = bool(dynamic), float(epsilon), bool(record)
        self.dev = torch.device(f"cuda:{device}")
        self.tdt = torch.float32 if dtype == "f32" else torch.float64
        self.fab = Fabrics(config=default_config(1), device=device)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev, dtype=self.tdt)
        self.state = t(np.concatenate([q0, qdot0], axis=2).transpose(2, 1, 0))              # (6,R,B)
        self.goal = t(goals.transpose(1, 2, 0))                                             # (R,2,B)
        self.weight = t(np.broadcast_to(np.asarray(weight, dtype=np.float64), (B, R)).T)    # (R,B)
        self.radius = t(np.broadcast_to(np.asarray(radius, dtype=np.float64), (B, R)).T)    # (R,B)
        self.scene = t(scene.transpose(1, 2, 0)) if self.S else None                       # (S,4,B)
        i32 = lambda v: torch.full((B,), v, dtype=torch.int32, device=self.dev)
        self.time_step, self.done_at, self.nonfinite_steps = i32(0), i32(-1), i32(0)
        self.min_clear_robots = torch.full((B,), float("inf"), dtype=self.tdt, device=self.dev)
        self.min_clear_scene = torch.full((B,), float("inf"), dtype=self.tdt, device=self.dev)
        self.traj = []                                                                      # (n,3,R,B) per run()
        self.steps_done = 0
        self._ep = None

    def _episode_struct(self):
        """The MrfPointEpisode argument of mrf_point_episode_run_dev_* (built once: the state tensors never move)."""
        import ctypes as C
        from ._lib import MrfPointEpisode
        ep = MrfPointEpisode()
        ep.struct_size = C.sizeof(MrfPointEpisode)
        ep.n_robots, ep.dynamic, ep.n_scene, ep.epsilon = self.R, int(self.dynamic), self.S, self.epsilon
        p = lambda t: None if t is None else t.data_ptr()
        ep.state, ep.goal, ep.weight, ep.radius, ep.scene = p(self.state), p(self.goal), p(self.weight), p(self.radius), p(self.scene)
        ep.time_step, ep.done_at, ep.nonfinite_steps = p(self.time_step), p(self.done_at), p(self.nonfinite_steps)
        ep.min_clear_robots, ep.min_clear_scene = p(self.min_clear_robots), p(self.min_clear_scene)
        return ep

    def run(self, n_steps: int):
        """n_steps control steps in one kernel launch on torch's current stream."""
        import ctypes as C
        from ._lib import check, lib
        if self._ep is None:
            self._ep = self._episode_struct()
        n_steps = int(n_steps)
        traj = None
        if self.record and n_steps > 0:
            traj = self.torch.empty((n_steps, 3, self.R, self.B), dtype=self.tdt, device=self.dev)
            self.traj.append(traj)
        self._ep.traj = None if traj is None else traj.data_ptr()
        fn = lib().mrf_point_episode_run_dev_f32 if self.tdt == self.torch.float32 else lib().mrf_point_episode_run_dev_f64
        check(fn(self.fab.handle.ptr, C.byref(self._ep), self.B, n_steps, self.torch.cuda.current_stream(self.dev).cuda_stream),
              "mrf_point_episode_run_dev")
        self.steps_done += n_steps
        return self

    def results(self) -> dict:
        """success, steps_to_success (-1 = not reached), min_clear_robots / min_clear_scene (running minima), nonfinite_steps
        (B,); q, qdot (B,R,3); traj (B,T,R,3), q after each step, when recorded."""
        self.torch.cuda.synchronize(self.dev)
        done = self.done_at.cpu().numpy()
        st = self.state.permute(2, 1, 0).double().cpu().numpy()                             # (B,R,6)
        out = {"steps": self.steps_done, "success": done >= 0, "steps_to_success": done,
               "min_clear_robots": self.min_clear_robots.double().cpu().numpy(),
               "min_clear_scene": self.min_clear_scene.double().cpu().numpy(),
               "nonfinite_steps": self.nonfinite_steps.cpu().numpy(), "q": st[:, :, 0:3], "qdot": st[:, :, 3:6]}
        if self.record:
            tr = self.torch.cat(self.traj) if self.traj else self.torch.empty((0, 3, self.R, self.B), dtype=self.tdt)
            out["traj"] = tr.permute(3, 0, 2, 1).double().cpu().numpy()
        return out
