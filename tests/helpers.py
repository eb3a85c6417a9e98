"""Shared helpers for the test-suite (oracle-side input preparation)."""
import numpy as np

from oracle import o2


def rel_ps(got, ref, ok=None):
    """Worst PER-SCENARIO relative error: for every scenario (axis 0) max |got - ref| over the remaining axes divided by
    that scenario's own max |ref|; the maximum over the scenarios selected by `ok`."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    ax = tuple(range(1, ref.ndim))
    e = np.abs(got - ref).max(axis=ax) / np.abs(ref).max(axis=ax)
    return float(e.max() if ok is None else e[ok].max())


def err_ps(got, ref):
    """PER-SCENARIO error with a unit floor: for every scenario (axis 0) max |got - ref| over the remaining axes divided by
    max(1, max |ref|) -- relative for large values, absolute for small ones.  A non-finite result counts as infinite."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    ax = tuple(range(1, ref.ndim))
    with np.errstate(invalid="ignore"):
        e = np.abs(got - ref).max(axis=ax) / np.maximum(1.0, np.abs(ref).max(axis=ax))
    return np.nan_to_num(e, nan=np.inf)


def oracle_rollout(rec, R, N, estimate_goal=0, static_or_dyn=1):
    """Oracle O2 coupled rollout incl. the RF-CV goal estimate; returns qN, qdN, avg, xee, goal_est, ok-mask."""
    ocfg = o2.default_config(R, static_or_dyn=static_or_dyn)
    rec_o = np.array(rec, dtype=np.float64, copy=True)
    B = rec_o.shape[0]
    goal = rec_o[:, 1, o2.G0:o2.G0 + 3].copy() if R > 1 else np.zeros((B, 3))
    if estimate_goal:
        for b in range(B):
            x, v = o2.endeffector(ocfg, 1, rec_o[b, 1, 0:7], rec_o[b, 1, 7:14], use_jqd=(estimate_goal == 2))
            goal[b] = x + 0.2 * v
        rec_o[:, 1, o2.G0:o2.G0 + 3] = goal
    lib = o2.lib()
    qN, qdN = np.zeros((B, R, N, 7)), np.zeros((B, R, N, 7))
    avg, xee = np.zeros((B, R)), np.zeros((B, R, 3))
    import ctypes as C
    lib.mrfo_rollout_jointspace_batch(C.byref(ocfg), o2._p(np.ascontiguousarray(rec_o)), B, N, o2._p(qN), o2._p(qdN),
                                      o2._p(avg), o2._p(xee), 0)
    mx = np.abs(qdN).max(axis=(1, 2, 3))
    ok = np.isfinite(mx) & (mx < 3.0)    # drop numerically stiff near-contact scenarios (blow-ups under dt = 0.01; see scenarios.py)
    return qN, qdN, avg, xee, goal, ok


def random_obstacles(rng, B, n_rob, S, rec=None, robot_first=0):
    """Random spheres; with `rec` (B,n_rob,44) those closer than a normalised clearance of 0.5 to any link of the ego
    robot are pushed up out of the workspace so the leaves stay well conditioned (0.02/x^4 metric)."""
    obst = np.zeros((B, n_rob, S, 10))
    obst[..., 0:3] = rng.uniform([-0.6, -1.2, 0.9], [1.6, 1.2, 2.0], size=(B, n_rob, S, 3))
    if rec is not None and S > 0:
        from multi_robot_fabrics_b200 import scenarios as sc
        for r in range(n_rob):
            pos = sc.link_positions(rec[:, r, 0:7], sc.mount_matrix(robot_first + r))          # B,8,3
            d = np.linalg.norm(obst[:, r, :, None, 0:3] - pos[:, None, :, :], axis=-1).min(axis=-1)   # B,S
            obst[:, r, :, 2] += np.where(d / 0.16 - 1.0 < 0.5, 1.5, 0.0)
    obst[..., 3:6] = rng.uniform(-0.3, 0.3, size=(B, n_rob, S, 3))
    obst[..., 6:9] = rng.uniform(-0.5, 0.5, size=(B, n_rob, S, 3))
    obst[..., 9] = 0.08
    return obst


def oracle_actions(rec, obst, robot_first=0, **cfgkw):
    """rec (B,n_rob,44), obst (B,n_rob,S,10) -> actions (B,n_rob,7) from oracle O2 (NaN rows where it fails)."""
    B, n_rob = rec.shape[:2]
    ocfg = o2.default_config(max(2, robot_first + n_rob), **cfgkw)
    out = np.full((B, n_rob, 7), np.nan)
    for b in range(B):
        for r in range(n_rob):
            o = obst[b, r]
            try:
                out[b, r] = o2.action(ocfg, robot_first + r, rec[b, r], o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9])
            except FloatingPointError:
                pass
    return out


def oracle_episode(rec, T, N, rollout=True, resolve=True, estimate=False, n_per_link=1):
    """CPU restatement of the closed control loop (examples/example_pandas_Jointspace.py:280-458) for ONE scenario with
    the reach-task protocol of multi_robot_fabrics_b200.episodes: oracle O2 + the deadlock restatement."""
    from oracle.deadlock_ref import DeadlockOracle
    R = rec.shape[0]
    cfg = o2.default_config(R)
    off = o2.sphere_offsets_ref(n_per_link)
    vlim = np.array([2.175] * 4 + [2.61] * 3)
    q, qd = rec[:, 0:7].copy(), rec[:, 7:14].copy()
    goal0, w0 = rec[:, 14:17].copy(), rec[:, 17].copy()
    dl, tdo, n_flags, done_at = DeadlockOracle(R), 1000, 0, -1
    for t in range(T):
        qd = np.clip(qd, -vlim, vlim)
        goals, weights = [g.copy() for g in goal0], list(w0)
        xee = [o2.kinematics(cfg, i, q[i], qd[i])[0][7] for i in range(R)]
        if rollout:
            if estimate:
                x, v = o2.endeffector(cfg, 1, q[1], qd[1])
                goals[1] = x + 0.2 * v
            r = rec.copy()
            r[:, 0:7], r[:, 7:14], r[:, 14:17], r[:, 17], r[:, 21] = q, qd, np.array(goals), weights, 10.0
            avg, _ = o2.rollout_jointspace_avg(cfg, r, N)
            if resolve:
                goals, weights, tdo, flag = dl.step(xee, goals, weights, t, tdo, float(sum(avg[0]) / R), [0] * R)
                n_flags += int(flag)
        lists = o2.obstacle_lists(cfg, q, qd, off, vel_mode=0)
        act = np.zeros((R, 7))
        for i in range(R):
            r = rec[i].copy()
            r[0:7], r[7:14], r[14:17], r[17], r[21] = q[i], qd[i], goals[i], weights[i], 20.0
            o = lists[i]
            act[i] = o2.action(cfg, i, r, o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9])
        a = np.clip(act, -vlim, vlim)
        qd = a
        q = q + 0.01 * a
        if done_at < 0 and all(np.linalg.norm(xee[i] - goal0[i]) < 0.05 for i in range(R)):
            done_at = t
    return q, n_flags, done_at


def oracle_pick_and_place(rec, blocks, start_goal, T, N, rollout=True, resolve=True, estimate=False, n_per_link=1):
    """CPU restatement of the pick-and-place control loop (examples/example_pandas_Jointspace.py:280-458) for ONE scenario
    with the kinematic environment of multi_robot_fabrics_b200.episodes: oracle O2, the deadlock restatement and the
    state-machine restatement (both pinned to the reference's classes).  blocks (n_blocks, R, 3), start_goal (R, 3).
    -> q (R,7), states (R,), blocks picked (R,), deadlock steps, done_at, q_grip (R,2)"""
    from oracle.deadlock_ref import DeadlockOracle
    from oracle.fsm_ref import FsmOracle
    R, nb = rec.shape[0], blocks.shape[0]
    cfg = o2.default_config(R)
    cfg_grasp = o2.default_config(R, has_collision_links=0)
    off = o2.sphere_offsets_ref(n_per_link)
    vlim = np.array([2.175] * 4 + [2.61] * 3)
    q, qd = rec[:, 0:7].copy(), rec[:, 7:14].copy()
    q_grip = np.full((R, 2), 0.04)
    fsm = [FsmOracle(start_goal[i], nb) for i in range(R)]
    goal_block = [np.zeros(3) for _ in range(R)]
    dl, tdo, n_flags, done_at = DeadlockOracle(R), 1000, 0, -1
    for t in range(T):
        qd = np.clip(qd, -vlim, vlim)
        xee = [o2.kinematics(cfg, i, q[i], qd[i])[0][7] for i in range(R)]
        for i in range(R):
            if fsm[i].n_ok < nb:
                goal_block[i] = blocks[fsm[i].n_ok, i] + np.array([0.0, 0.0, 0.1])                  # :302-303
        states = [fsm[i].step(xee[i], q_grip[i], goal_block[i]) for i in range(R)]
        if done_at < 0 and all(s == 10 for s in states):
            done_at = t
        goals, weights = [fsm[i].goal.copy() for i in range(R)], [float(fsm[i].weight) for i in range(R)]
        if rollout:
            if estimate:
                x, v = o2.endeffector(cfg, 1, q[1], qd[1])
                goals[1] = x + 0.2 * v
            r = rec.copy()
            r[:, 0:7], r[:, 7:14], r[:, 14:17], r[:, 17], r[:, 21] = q, qd, np.array(goals), weights, 10.0
            avg, _ = o2.rollout_jointspace_avg(cfg, r, N)
            if resolve:
                goals, weights, tdo, flag = dl.step(xee, goals, weights, t, tdo, float(sum(avg[0]) / R), list(states))
                n_flags += int(flag)
        lists = o2.obstacle_lists(cfg, q, qd, off, vel_mode=0)
        act = np.zeros((R, 7))
        for i in range(R):
            if states[i] in (3, 5):
                continue                                                                              # :418-419
            r = rec[i].copy()
            r[0:7], r[7:14], r[14:17], r[17], r[21] = q[i], qd[i], goals[i], weights[i], 20.0
            o = lists[i]
            try:
                act[i] = o2.action(cfg_grasp if states[i] == 2 else cfg, i, r, o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9])
            except FloatingPointError:          # metric not positive definite: NaN action, the arm holds still
                act[i] = np.nan
        a = np.clip(act, -vlim, vlim)
        a[~np.isfinite(a)] = 0.0
        for i in range(R):
            q_grip[i] = np.clip(q_grip[i] + 0.01 * fsm[i].gripper_action(q_grip[i]), 0.0, 0.04)
        qd = a
        q = q + 0.01 * a
    return q, np.array([f.state for f in fsm]), np.array([f.n_ok for f in fsm]), n_flags, done_at, q_grip
