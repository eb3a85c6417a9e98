"""Self-collision leaves on top of the oracles, for the tests (fabrics set_components(..., self_collision_pairs)).

A pair (a, b) of one robot's links is the 1-D leaf x = |p_a - p_b| / rho - 1 with
    Finsler energy L = k_f s_f xdot^2 / x^p_f,  geometry h = k_g s_g xdot^2 / x^p_g,  s = -0.5 (sign(xdot) - 1) if gated.
Two independent restatements of its contribution (M_q, f_q, f_e,q) to the planner's geometry:
  - `o1_pair_terms`: autodiff, oracle O1's `_static_leaf` on phi(q) = |fk_a(q) - fk_b(q)| / rho - 1 with the leaf as a
    fabrics expression string;
  - `closed_pair_terms`: the closed form the kernels use (the sphere leaf on the relative point, columns J_a - J_b).
Either is added to the diagnostics of an oracle action (O1 `action_raw` or O2 `action(want_diag=True)`) and
`finish_action` repeats the planner's solve and damper on the sums.  Link numbers: 1..8 = panda_linkN, 9 = panda_hand.
"""
import numpy as np
import torch

from oracle import o1_fabrics as o1

LINK_NAMES = {**{l: f"panda_link{l}" for l in range(1, 9)}, 9: "panda_hand"}
# fabrics 0.9.5 self_collision_geometry / self_collision_finsler as recalled (DESIGN.md A13)
DEFAULT_LEAF = dict(k_geometry=-0.5, p_geometry=1, gate_geometry=1, k_finsler=0.1, p_finsler=2, gate_finsler=0)


def leaf_strings(leaf=None):
    """The leaf as fabrics expression strings (geometry, finsler)."""
    c = {**DEFAULT_LEAF, **(leaf or {})}
    gate = " * (-0.5 * (ca.sign(xdot) - 1))"
    geo = f"{c['k_geometry']!r} / (x ** {c['p_geometry']}){gate if c['gate_geometry'] else ''} * xdot ** 2"
    fin = f"{c['k_finsler']!r} / (x ** {c['p_finsler']}){gate if c['gate_finsler'] else ''} * xdot ** 2"
    return geo, fin


def o1_pair_terms(q, qd, mount, pairs, rho, leaf=None, jdot_sign=-1.0):
    """Sum over the pairs of (M_q, f_q, f_e,q) by autodiff (oracle O1)."""
    geo, fin = leaf_strings(leaf)
    pl = o1.O1Planner(7, lambda qq, link: o1.panda_fk(qq, mount, link), o1.FabricConfig(jdot_sign=jdot_sign))
    t = lambda v: torch.as_tensor(np.asarray(v, dtype=np.float64), dtype=torch.float64)
    q, qd = t(q), t(qd)
    M, f, fe = np.zeros((7, 7)), np.zeros(7), np.zeros(7)
    for (a, b), r in zip(pairs, rho):
        la, lb = LINK_NAMES[a], LINK_NAMES[b]
        phi = lambda qq, la=la, lb=lb, r=float(r): (torch.sqrt(((o1.panda_fk(qq, mount, la) - o1.panda_fk(qq, mount, lb)) ** 2)
                                                                .sum()) / r - 1.0).reshape(1)
        Mq, fq, feq = pl._static_leaf(q, qd, phi, geo, fin)
        M, f, fe = M + Mq.numpy(), f + fq.numpy(), fe + feq.numpy()
    return M, f, fe


def o2_kin(ocfg, robot):
    """Point kinematics from oracle O2: link l -> x, v = J qdot, c = d(J qdot)/dq qdot, J (panda_hand = link 8)."""
    from oracle import o2

    def kin(q, qd):
        x, v, c, J = o2.kinematics(ocfg, robot, q, qd)
        return lambda l: (x[min(l, 8) - 1], v[min(l, 8) - 1], c[min(l, 8) - 1], J[min(l, 8) - 1])
    return kin


def closed_pair_terms(q, qd, mount, pairs, rho, leaf=None, jdot_sign=-1.0, kin_of=None):
    """The same sums in closed form (the kernels' arrangement); point kinematics x, J, d(J qdot)/dq qdot from O1's FK,
    or from `kin_of(q, qd)` (e.g. `o2_kin(ocfg, robot)`)."""
    c = {**DEFAULT_LEAF, **(leaf or {})}
    M, f, fe = np.zeros((7, 7)), np.zeros(7), np.zeros(7)
    kin = {}
    k2 = kin_of(q, qd) if kin_of is not None else None
    for (a, b), r in zip(pairs, rho):
        for l in (a, b):
            if l not in kin:
                kin[l] = k2(l) if k2 is not None else o1.link_kinematics(q, qd, mount, LINK_NAMES[l], jdot_ref_sign=1.0)
        xa, va, ca, Ja = kin[a]
        xb, vb, cb, Jb = kin[b]
        d, w, cr, J = xa - xb, va - vb, ca - cb, Ja - Jb
        n = np.sqrt(d @ d)
        gs = 1.0 / (n * r)
        x = n / r - 1.0
        xd = (d @ w) * gs
        s = 0.0 if xd > 0 else (1.0 if xd < 0 else 0.5)
        Ml = 2.0 * c["k_finsler"] * (s if c["gate_finsler"] else 1.0) / x ** c["p_finsler"]
        hh = c["k_geometry"] * (s if c["gate_geometry"] else 1.0) / x ** c["p_geometry"]
        # J-dot qdot of x: gs (|w|^2 + d.c) - (d.w)^2 gs / n^2, with fabrics' sign on the whole term
        xdd = gs * (w @ w + d @ cr) - (d @ w) ** 2 * gs / (n * n)
        u = J.T @ d * gs                                   # dx/dq
        M += Ml * np.outer(u, u)
        f += u * (Ml * hh * xd * xd + Ml * jdot_sign * xdd)
        fe += u * (-0.5 * c["p_finsler"] * Ml * xd * xd / x + Ml * xdd)
    return M, f, fe


def finish_action(q, qd, x_goal_0, p_hand, M_g, f_g, fe_g, M_f, f_f, mode="vel", dt=0.01, eps=1e-6, exec_scale=1.0):
    """O1Planner.action_raw from the summed specs on: solves, speed-control damper, 'vel' / 'acc' output."""
    e = eps
    I = np.eye(7)
    h_g = np.linalg.solve(M_g + e * I, f_g)
    h_f = np.linalg.solve(M_f + e * I, f_f)
    a_geom = -(qd @ (f_g - fe_g)) / (e + qd @ (M_g @ qd))
    s2 = 2.0 * exec_scale
    den = e + s2 * (qd @ qd)
    a_ex0, a_exf = -(qd @ (s2 * h_g)) / den, -(qd @ (s2 * h_f)) / den
    eta = 0.5 * (np.tanh(-0.9 * 0.5 * (qd @ qd) - 0.5) + 1.0)
    a_ex = eta * a_ex0 + (1.0 - eta) * a_exf
    xpsi = np.linalg.norm(p_hand - x_goal_0)
    beta = 0.5 * (np.tanh(-0.5 * (xpsi - 0.02)) + 1.0) * 6.5 + 0.01 + max(0.0, a_geom - a_ex)
    qdd = -h_f - (a_ex + beta) * qd
    return qd + dt * qdd if mode == "vel" else qdd


def action_with_pairs(diag, rec, mount, pairs, rho, leaf=None, terms=closed_pair_terms, mode="vel", dt=0.01, ocfg=None,
                      robot=None):
    """An oracle action's diagnostics (M_g, f_g, fe_g, M_f, f_f) plus the pair leaves -> the action of the planner with
    self-collision.  rec: the robot's 44-scalar record.  With ocfg / robot the closed form takes O2's kinematics."""
    q, qd = np.asarray(rec[0:7], dtype=np.float64), np.asarray(rec[7:14], dtype=np.float64)
    if ocfg is not None:
        from oracle import o2
        M, f, fe = closed_pair_terms(q, qd, mount, pairs, rho, leaf, kin_of=o2_kin(ocfg, robot)) if pairs else (0.0, 0.0, 0.0)
        p_hand = o2.kinematics(ocfg, robot, q, qd)[0][7]
    else:
        M, f, fe = terms(q, qd, mount, pairs, rho, leaf) if pairs else (0.0, 0.0, 0.0)
        p_hand = o1.panda_fk(torch.as_tensor(q), mount, "panda_hand").numpy()
    return finish_action(q, qd, np.asarray(rec[14:17]), p_hand, diag["M_g"] + M, diag["f_g"] + f, diag["fe_g"] + fe,
                         diag["M_f"] + M, diag["f_f"] + f, mode=mode, dt=dt)


def coupled_rollout(ocfg, rec, N, pairs, rho, leaf=None):
    """The coupled rollout (forward_planner_Jointspace.py:190-249, 'vel' mode) of one scenario, rec (R,44), with each
    robot's pairs: step with the stale velocity, publish every robot's links, then every action against the other
    robots' links as moving spheres.  Returns qN, qdN (R,N,7)."""
    from oracle import o2
    R = ocfg.n_robots
    q = [np.array(rec[r, 0:7], dtype=np.float64) for r in range(R)]
    qd = [np.array(rec[r, 7:14], dtype=np.float64) for r in range(R)]
    qN, qdN = np.zeros((R, N, 7)), np.zeros((R, N, 7))
    mounts = [o2.mount_of(ocfg, r) for r in range(R)]
    for k in range(N):
        for r in range(R):
            q[r] = q[r] + ocfg.dt * qd[r]
        kin = [o2.kinematics(ocfg, r, q[r], qd[r]) for r in range(R)]
        new = []
        for r in range(R):
            others = [j for j in range(R) if j != r]
            xo = np.array([kin[j][0] for j in others]).reshape(-1, 3)
            vo = np.array([kin[j][1] for j in others]).reshape(-1, 3)
            ao = ocfg.jdot_ref_sign * np.array([kin[j][2] for j in others]).reshape(-1, 3)  # a = J qdd + Jdot qdot, qdd = 0
            ro = np.array([ocfg.r_robots[j][:] for j in others]).reshape(-1)
            cur = np.array(rec[r], dtype=np.float64)
            cur[0:7], cur[7:14] = q[r], qd[r]
            _, d = o2.action(ocfg, r, cur, xo, vo, ao, ro, want_diag=True)
            new.append(action_with_pairs(d, cur, mounts[r], pairs[r] if r < len(pairs) else [],
                                         rho[r] if r < len(rho) else [], leaf, ocfg=ocfg, robot=r))
        for r in range(R):
            qd[r] = new[r]
            qN[r, k], qdN[r, k] = q[r], qd[r]
    return qN, qdN


def o1_coupled_rollout(ocfg, rec, N, pairs, rho, leaf=None):
    """The same coupled rollout with oracle O1 throughout: autodiff planner (`action_raw`), autodiff pair leaves and O1's
    link kinematics for the published spheres.  Returns qN, qdN (R,N,7)."""
    from oracle import o2
    R = ocfg.n_robots
    mounts = [o2.mount_of(ocfg, r) for r in range(R)]
    planners = [o1.make_panda_planner(mounts[r], n_dyn=8 * (R - 1)) for r in range(R)]
    q = [np.array(rec[r, 0:7], dtype=np.float64) for r in range(R)]
    qd = [np.array(rec[r, 7:14], dtype=np.float64) for r in range(R)]
    qN, qdN = np.zeros((R, N, 7)), np.zeros((R, N, 7))
    for k in range(N):
        for r in range(R):
            q[r] = q[r] + ocfg.dt * qd[r]
        kin = [[o1.link_kinematics(q[r], qd[r], mounts[r], f"panda_link{l}", ocfg.jdot_ref_sign)[:3] for l in range(1, 9)]
               for r in range(R)]
        new = []
        for r in range(R):
            p = o2.record_to_params(rec[r])
            o = 0
            for j in range(R):
                if j == r:
                    continue
                for l in range(8):
                    x, v, a = kin[j][l]
                    p[f"x_obst_dynamic_{o}"], p[f"xdot_obst_dynamic_{o}"], p[f"xddot_obst_dynamic_{o}"] = x, v, a
                    p[f"radius_obst_dynamic_{o}"] = ocfg.r_robots[j][l]
                    o += 1
            cur = np.array(rec[r], dtype=np.float64)
            cur[0:7], cur[7:14] = q[r], qd[r]
            _, d = planners[r].action_raw(q[r], qd[r], p)
            new.append(action_with_pairs(d, cur, mounts[r], pairs[r], rho[r], leaf, terms=o1_pair_terms))
        for r in range(R):
            qd[r] = new[r]
            qN[r, k], qdN[r, k] = q[r], qd[r]
    return qN, qdN


def cartesian_rollout(ocfg, robot, rec, obst, N, pairs, rho, leaf=None, use_o1=False):
    """Decoupled Cartesian rollout (forward_planner_Cartesian.py:421-458, 'vel' mode) of one robot against spheres at
    constant velocity, obst (S,10) with zero accelerations; O2 + closed form, or O1 + autodiff.  Returns qdN (N,7)."""
    from oracle import o2
    mount = o2.mount_of(ocfg, robot)
    pl = o1.make_panda_planner(mount, n_dyn=len(obst)) if use_o1 else None
    cur = np.array(rec, dtype=np.float64)
    xo = obst[:, 0:3].copy()
    out = np.zeros((N, 7))
    for k in range(N):
        if use_o1:
            p = o2.record_to_params(cur)
            for i in range(len(obst)):
                p[f"x_obst_dynamic_{i}"], p[f"xdot_obst_dynamic_{i}"] = xo[i], obst[i, 3:6]
                p[f"xddot_obst_dynamic_{i}"], p[f"radius_obst_dynamic_{i}"] = np.zeros(3), obst[i, 9]
            _, d = pl.action_raw(cur[0:7], cur[7:14], p)
            qd = action_with_pairs(d, cur, mount, pairs, rho, leaf, terms=o1_pair_terms)
        else:
            _, d = o2.action(ocfg, robot, cur, xo, obst[:, 3:6], obst[:, 6:9], obst[:, 9], want_diag=True)
            qd = action_with_pairs(d, cur, mount, pairs, rho, leaf, ocfg=ocfg, robot=robot)
        cur[7:14] = qd
        cur[0:7] = cur[0:7] + ocfg.dt * qd
        xo = xo + ocfg.dt * obst[:, 3:6]
        out[k] = qd
    return out


VLIM = np.array([2.175] * 4 + [2.61] * 3)


def _rollout_avg(cfg, r, N, pairs, rho):
    _, qdN = coupled_rollout(cfg, r, N, pairs, rho)
    return (qdN ** 2).sum(axis=(1, 2)) / (N * 7)


def episode(rec, T, N, pairs, rho, rollout=True, resolve=True, estimate=False, n_per_link=1):
    """tests/helpers.oracle_episode (the reach-task control loop on the CPU with O2 and the deadlock restatement) with
    each robot's self-collision pairs in the rollouts and the executed actions.  -> q (R,7), deadlock steps, done_at."""
    from oracle import o2
    from oracle.deadlock_ref import DeadlockOracle
    R = rec.shape[0]
    cfg = o2.default_config(R)
    off = o2.sphere_offsets_ref(n_per_link)
    q, qd = rec[:, 0:7].copy(), rec[:, 7:14].copy()
    goal0, w0 = rec[:, 14:17].copy(), rec[:, 17].copy()
    dl, tdo, n_flags, done_at = DeadlockOracle(R), 1000, 0, -1
    for t in range(T):
        qd = np.clip(qd, -VLIM, VLIM)
        goals, weights = [g.copy() for g in goal0], list(w0)
        xee = [o2.kinematics(cfg, i, q[i], qd[i])[0][7] for i in range(R)]
        if rollout:
            if estimate:
                x, v = o2.endeffector(cfg, 1, q[1], qd[1])
                goals[1] = x + 0.2 * v
            r = rec.copy()
            r[:, 0:7], r[:, 7:14], r[:, 14:17], r[:, 17], r[:, 21] = q, qd, np.array(goals), weights, 10.0
            avg = _rollout_avg(cfg, r, N, pairs, rho)
            if resolve:
                goals, weights, tdo, flag = dl.step(xee, goals, weights, t, tdo, float(sum(avg) / R), [0] * R)
                n_flags += int(flag)
        lists = o2.obstacle_lists(cfg, q, qd, off, vel_mode=0)
        act = np.zeros((R, 7))
        for i in range(R):
            r = rec[i].copy()
            r[0:7], r[7:14], r[14:17], r[17], r[21] = q[i], qd[i], goals[i], weights[i], 20.0
            o = lists[i]
            _, d = o2.action(cfg, i, r, o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9], want_diag=True)
            act[i] = action_with_pairs(d, r, o2.mount_of(cfg, i), pairs[i], rho[i], ocfg=cfg, robot=i)
        a = np.clip(act, -VLIM, VLIM)
        qd = a
        q = q + 0.01 * a
        if done_at < 0 and all(np.linalg.norm(xee[i] - goal0[i]) < 0.05 for i in range(R)):
            done_at = t
    return q, n_flags, done_at


def pick_and_place(rec, blocks, start_goal, T, N, pairs, rho, rollout=True, resolve=True, n_per_link=1):
    """tests/helpers.oracle_pick_and_place with each robot's self-collision pairs in the rollouts and in both executed
    planners (the grasp planner of state 2 included).  -> q (R,7), states (R,), blocks picked (R,), deadlock steps,
    done_at, q_grip (R,2)"""
    from oracle import o2
    from oracle.deadlock_ref import DeadlockOracle
    from oracle.fsm_ref import FsmOracle
    R, nb = rec.shape[0], blocks.shape[0]
    cfg = o2.default_config(R)
    cfg_grasp = o2.default_config(R, has_collision_links=0)
    off = o2.sphere_offsets_ref(n_per_link)
    q, qd = rec[:, 0:7].copy(), rec[:, 7:14].copy()
    q_grip = np.full((R, 2), 0.04)
    fsm = [FsmOracle(start_goal[i], nb) for i in range(R)]
    goal_block = [np.zeros(3) for _ in range(R)]
    dl, tdo, n_flags, done_at = DeadlockOracle(R), 1000, 0, -1
    seen = set()
    for t in range(T):
        qd = np.clip(qd, -VLIM, VLIM)
        xee = [o2.kinematics(cfg, i, q[i], qd[i])[0][7] for i in range(R)]
        for i in range(R):
            if fsm[i].n_ok < nb:
                goal_block[i] = blocks[fsm[i].n_ok, i] + np.array([0.0, 0.0, 0.1])
        states = [fsm[i].step(xee[i], q_grip[i], goal_block[i]) for i in range(R)]
        seen.update(states)
        if done_at < 0 and all(s == 10 for s in states):
            done_at = t
        goals, weights = [fsm[i].goal.copy() for i in range(R)], [float(fsm[i].weight) for i in range(R)]
        if rollout:
            r = rec.copy()
            r[:, 0:7], r[:, 7:14], r[:, 14:17], r[:, 17], r[:, 21] = q, qd, np.array(goals), weights, 10.0
            avg = _rollout_avg(cfg, r, N, pairs, rho)
            if resolve:
                goals, weights, tdo, flag = dl.step(xee, goals, weights, t, tdo, float(sum(avg) / R), list(states))
                n_flags += int(flag)
        lists = o2.obstacle_lists(cfg, q, qd, off, vel_mode=0)
        act = np.zeros((R, 7))
        for i in range(R):
            if states[i] in (3, 5):
                continue
            r = rec[i].copy()
            r[0:7], r[7:14], r[14:17], r[17], r[21] = q[i], qd[i], goals[i], weights[i], 20.0
            o = lists[i]
            c = cfg_grasp if states[i] == 2 else cfg
            try:
                _, d = o2.action(c, i, r, o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9], want_diag=True)
                act[i] = action_with_pairs(d, r, o2.mount_of(cfg, i), pairs[i], rho[i], ocfg=cfg, robot=i)
            except (FloatingPointError, np.linalg.LinAlgError):
                act[i] = np.nan
        a = np.clip(act, -VLIM, VLIM)
        a[~np.isfinite(a)] = 0.0
        for i in range(R):
            q_grip[i] = np.clip(q_grip[i] + 0.01 * fsm[i].gripper_action(q_grip[i]), 0.0, 0.04)
        qd = a
        q = q + 0.01 * a
    return q, np.array([f.state for f in fsm]), np.array([f.n_ok for f in fsm]), n_flags, done_at, q_grip, seen
