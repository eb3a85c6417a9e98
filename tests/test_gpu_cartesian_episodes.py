"""GPU tests of the decoupled Cartesian rollout model: the all-robot rollout entry (mrf_rollout_cart_all_dev) and the
closed control loop of examples/example_pandas_cartesian.py (BatchedEpisodes(rollouts="cartesian")), against per-robot
calls of the single-robot entry and against the same loop run on the CPU with oracle O2 and the deadlock / state-machine
restatements."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200._lib import MrfError
from multi_robot_fabrics_b200.api import Fabrics, to_soa
from oracle import o2

from helpers import rel_ps

VLIM = np.array([2.175] * 4 + [2.61] * 3)


def same_bits(a, b):
    """Bitwise equality of two float tensors, NaN payloads included (a few random scenarios blow up under dt = 0.01)."""
    import torch
    it = torch.int64 if a.dtype == torch.float64 else torch.int32
    return torch.equal(a.contiguous().view(it), b.contiguous().view(it))


def _cart_avg(cfg, rec, q, qd, goals, weights, off, N):
    """Rollout step of the Cartesian loop: every robot rolled out alone (weight_goal_1 = 20) against the other robots'
    spheres with their true velocities, moving at constant velocity (example_pandas_cartesian.py:343-418)."""
    R = len(q)
    lists = o2.obstacle_lists(cfg, q, qd, off, vel_mode=1)
    avg = np.zeros(R)
    for i in range(R):
        r = rec[i].copy()
        r[0:7], r[7:14], r[14:17], r[17], r[21] = q[i], qd[i], goals[i], weights[i], 20.0
        o = lists[i]
        avg[i] = o2.rollout_cartesian(cfg, i, r, o[:, 0:3], o[:, 3:6], o[:, 9], N)[2]
    return avg


def oracle_cartesian_episode(rec, T, N, resolve=True, estimate=False, n_per_link=1):
    """CPU restatement of the Cartesian control loop (examples/example_pandas_cartesian.py:295-462) for ONE scenario with
    the reach-task protocol of multi_robot_fabrics_b200.episodes.  -> q (R,7), deadlock steps, done_at"""
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
        if estimate:                                                         # :355-357, true J qdot
            x, v = o2.endeffector(cfg, 1, q[1], qd[1], use_jqd=True)
            goals[1] = x + 0.2 * v
        avg = _cart_avg(cfg, rec, q, qd, goals, weights, off, N)
        if resolve:
            goals, weights, tdo, flag = dl.step(xee, goals, weights, t, tdo, float(sum(avg) / R), [0] * R)
            n_flags += int(flag)
        lists = o2.obstacle_lists(cfg, q, qd, off, vel_mode=0)
        act = np.zeros((R, 7))
        for i in range(R):
            r = rec[i].copy()
            r[0:7], r[7:14], r[14:17], r[17], r[21] = q[i], qd[i], goals[i], weights[i], 20.0
            o = lists[i]
            act[i] = o2.action(cfg, i, r, o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9])
        a = np.clip(act, -VLIM, VLIM)
        qd = a
        q = q + 0.01 * a
        if done_at < 0 and all(np.linalg.norm(xee[i] - goal0[i]) < 0.05 for i in range(R)):
            done_at = t
    return q, n_flags, done_at


def oracle_cartesian_pick_and_place(rec, blocks, start_goal, T, N, resolve=True, estimate=False, n_per_link=1):
    """The pick-and-place protocol of helpers.oracle_pick_and_place with the Cartesian rollout step.
    -> q (R,7), states (R,), blocks picked (R,), deadlock steps, done_at, q_grip (R,2)"""
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
    for t in range(T):
        qd = np.clip(qd, -VLIM, VLIM)
        xee = [o2.kinematics(cfg, i, q[i], qd[i])[0][7] for i in range(R)]
        for i in range(R):
            if fsm[i].n_ok < nb:
                goal_block[i] = blocks[fsm[i].n_ok, i] + np.array([0.0, 0.0, 0.1])
        states = [fsm[i].step(xee[i], q_grip[i], goal_block[i]) for i in range(R)]
        if done_at < 0 and all(s == 10 for s in states):
            done_at = t
        goals, weights = [fsm[i].goal.copy() for i in range(R)], [float(fsm[i].weight) for i in range(R)]
        if estimate:
            x, v = o2.endeffector(cfg, 1, q[1], qd[1], use_jqd=True)
            goals[1] = x + 0.2 * v
        avg = _cart_avg(cfg, rec, q, qd, goals, weights, off, N)
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
            try:
                act[i] = o2.action(cfg_grasp if states[i] == 2 else cfg, i, r, o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9])
            except FloatingPointError:
                act[i] = np.nan
        a = np.clip(act, -VLIM, VLIM)
        a[~np.isfinite(a)] = 0.0
        for i in range(R):
            q_grip[i] = np.clip(q_grip[i] + 0.01 * fsm[i].gripper_action(q_grip[i]), 0.0, 0.04)
        qd = a
        q = q + 0.01 * a
    return q, np.array([f.state for f in fsm]), np.array([f.n_ok for f in fsm]), n_flags, done_at, q_grip


def reach_scenarios(B, R, seed, offset):
    """Random reach tasks.  Every other scenario starts with the hands of robots 0 and 1 less than 0.35 m apart (drawn
    from a larger pool) and gives both nearly the same goal between them: the hands crowd each other and slow down, the
    situation the deadlock heuristic is there for."""
    sc = m.scenarios
    rec = sc.generate(B, R, seed=seed)
    pool = sc.generate(100 * B, R, seed=seed + 1)
    hand = [sc.link_positions(pool[:, r, 0:7], sc.mount_matrix(r))[:, 7] for r in range(2)]
    close = np.nonzero(np.linalg.norm(hand[0] - hand[1], axis=1) < 0.35)[0][: len(rec[1::2])]
    rec[1::2] = pool[close]
    mid = 0.5 * (hand[0][close] + hand[1][close])
    rec[1::2, 0, 14:17] = mid
    rec[1::2, 1, 14:17] = mid + offset
    rec[:, :, 7:14] *= 0.2
    return rec


@pytest.mark.parametrize("R", [2, 3])
def test_rollout_cart_all_matches_per_robot_calls_and_oracle(built, R):
    """One launch for every robot == R calls of the single-robot entry on the per-robot slices, bit for bit (FP64 and
    FP32); FP64 == oracle O2's decoupled rollout."""
    import torch
    B, N, n = 64, 10, 2
    S = 8 * n * (R - 1)
    rec = m.scenarios.generate(B, R, seed=81, weight_goal_1=20.0)
    rec[:, :, 7:14] *= 0.3
    fab = Fabrics(R, device=0)
    dev = "cuda:0"
    for dt in (torch.float64, torch.float32):
        d = torch.from_numpy(to_soa(rec)).to(dev, dtype=dt)
        obst = fab.obstacles_dev(d[0:7].contiguous(), d[7:14].contiguous(), n_per_link=n, vel_mode=1)
        assert obst.shape == (S, 10, R, B)
        qN = torch.empty((R, N, 7, B), dtype=dt, device=dev)
        qdN = torch.empty_like(qN)
        avg = fab.rollout_cart_all_dev(d, obst, N, qN=qN, qdN=qdN)
        for r in range(R):
            q1, qd1 = torch.empty((N, 7, B), dtype=dt, device=dev), torch.empty((N, 7, B), dtype=dt, device=dev)
            a1 = fab.rollout_cart_dev(r, d[:, r].contiguous(), obst[:, :, r].contiguous(), N, qN=q1, qdN=qd1)
            torch.cuda.synchronize()
            assert same_bits(avg[r], a1) and same_bits(qN[r], q1) and same_bits(qdN[r], qd1), (dt, r)
        if dt != torch.float64:
            continue
        o = obst.permute(3, 2, 0, 1).cpu().numpy()                                     # (B,R,S,10)
        got_q, got_qd = qN.permute(3, 0, 1, 2).cpu().numpy(), qdN.permute(3, 0, 1, 2).cpu().numpy()
        got_a = avg.T.cpu().numpy()
        ocfg = o2.default_config(R)
        ref_q, ref_qd, ref_a = np.zeros((B, R, N, 7)), np.zeros((B, R, N, 7)), np.zeros((B, R))
        for b in range(B):
            for r in range(R):
                ref_q[b, r], ref_qd[b, r], ref_a[b, r] = o2.rollout_cartesian(
                    ocfg, r, rec[b, r], o[b, r, :, 0:3], o[b, r, :, 3:6], o[b, r, :, 9], N)
        mx = np.abs(ref_qd).max(axis=(1, 2, 3))
        ok = np.isfinite(mx) & (mx < 3.0)
        assert ok.sum() >= B - 8
        assert rel_ps(got_q, ref_q, ok) < 1e-9 and rel_ps(got_qd, ref_qd, ok) < 1e-9 and rel_ps(got_a, ref_a, ok) < 1e-9
    fab.close()


@pytest.mark.parametrize("R,estimate", [(2, True), (3, False)])
def test_cartesian_episodes_match_cpu_loop(built, R, estimate):
    """The fused control step with decoupled Cartesian rollouts (captured in a CUDA graph) reproduces the Cartesian loop
    run on the CPU oracle, scenario by scenario, deadlock flags included.  R = 3 is the case the reference's own
    Cartesian example cannot run."""
    from multi_robot_fabrics_b200.episodes import BatchedEpisodes
    B, T, N = 12, 25, 5
    rec = reach_scenarios(B, R, 71, [0.05, 0.0, 0.02])
    ep = BatchedEpisodes(rec, n_horizon=N, dtype="f64", n_obst_per_link=2, rollouts="cartesian", estimate_goal=estimate)
    res = ep.run(T).results()
    n_cmp, flags = 0, 0
    for b in range(B):
        try:
            q, n_flags, done_at = oracle_cartesian_episode(rec[b], T, N, estimate=estimate, n_per_link=2)
        except FloatingPointError:
            continue
        if not np.isfinite(q).all():
            continue
        n_cmp += 1
        flags += n_flags
        assert np.abs(res["q"][b] - q).max() < 1e-7, b
        assert res["deadlock_steps"][b] == n_flags and res["steps_to_success"][b] == done_at, b
        assert res["nonfinite_steps"][b] == 0
    assert n_cmp >= B - 3 and res["steps"] == T
    assert flags > 0                       # the deadlock heuristic really fired on the compared scenarios


def test_cartesian_pick_and_place_matches_cpu_loop(built):
    """Pick-and-place protocol with Cartesian rollouts, RF-CV goal estimate and deadlock resolution against the CPU loop."""
    from multi_robot_fabrics_b200.episodes import BatchedEpisodes
    R, B, T, N, nb = 2, 4, 420, 3, 1
    rng = np.random.default_rng(9)
    rec = m.scenarios.generate(B, R, seed=91)
    rec[:, :, 7:14] = 0.0
    cfg = o2.default_config(R)
    start = np.zeros((B, R, 3))
    blocks = np.zeros((B, nb, R, 3))
    for b in range(B):
        for r in range(R):
            start[b, r] = o2.kinematics(cfg, r, rec[b, r, 0:7], rec[b, r, 7:14])[0][7]
            blocks[b, 0, r] = start[b, r] + np.array([rng.uniform(-0.06, 0.06), rng.uniform(-0.06, 0.06), -0.16])
    ep = BatchedEpisodes(rec, n_horizon=N, dtype="f64", n_obst_per_link=1, blocks=blocks, start_goal=start,
                         rollouts="cartesian", estimate_goal=True)
    res = ep.run(T).results()
    for b in range(B):
        q, states, picked, n_flags, done_at, q_grip = oracle_cartesian_pick_and_place(rec[b], blocks[b], start[b], T, N,
                                                                                       estimate=True)
        assert np.array_equal(res["state"][b], states) and np.array_equal(res["blocks_picked"][b], picked), b
        assert res["steps_to_success"][b] == done_at and res["deadlock_steps"][b] == n_flags
        assert np.abs(res["q"][b] - q).max() < 1e-6 and np.abs(res["q_grip"][b] - q_grip).max() < 1e-12
    assert res["blocks_picked"].sum() > 0


@pytest.mark.parametrize("R,pnp", [(2, False), (3, False), (2, True)])
def test_cartesian_episodes_fp32_graph_equals_eager(built, R, pnp):
    """FP32: the graph-replayed control loop is bitwise the loop launched step by step."""
    from multi_robot_fabrics_b200.episodes import BatchedEpisodes
    B, T, N = 512, 40, 10
    rec = reach_scenarios(B, R, 72, [0.05, 0.0, 0.02])
    task = {}
    if pnp:
        rec[:, :, 7:14] = 0.0
        blocks, start = m.scenarios.pick_and_place_layout(rec, n_blocks=1, seed=1)
        task = dict(blocks=blocks, start_goal=start)
    runs = [BatchedEpisodes(rec, n_horizon=N, dtype="f32", rollouts="cartesian", estimate_goal=True, use_graph=g,
                            **task).run(T).results() for g in (True, False)]
    for k in ("q", "x_ee", "deadlock_steps", "steps_to_success", "min_clearance", "nonfinite_steps"):
        assert np.array_equal(runs[0][k], runs[1][k], equal_nan=k in ("q", "x_ee", "min_clearance")), k
    assert runs[0]["steps"] == runs[1]["steps"] == T


def test_cartesian_argument_checks(built):
    import ctypes as C
    import torch
    from multi_robot_fabrics_b200._lib import check, lib
    from multi_robot_fabrics_b200.episodes import BatchedEpisodes
    R, B = 2, 8
    rec = m.scenarios.generate(B, R, seed=73)
    with pytest.raises(MrfError):
        BatchedEpisodes(rec, rollouts="cartesian", rollout_fabrics=False)
    with pytest.raises(MrfError):
        BatchedEpisodes(rec, rollouts="taskspace")
    ep = BatchedEpisodes(rec, n_horizon=3, dtype="f64", rollouts="cartesian", use_graph=False)
    ep.run(1)
    st = ep._episode_struct()
    step = lambda: check(lib().mrf_episode_step_dev_f64(ep.fab.handle.ptr, C.byref(st), B,
                                                         torch.cuda.current_stream().cuda_stream), "mrf_episode_step_dev")
    st.rollout_model = 2
    with pytest.raises(MrfError, match="rollout_model"):
        step()
    st.rollout_model, st.kin_scratch = 1, None
    with pytest.raises(MrfError, match="kin_scratch"):
        step()
    st.rollout_fabrics, st.kin_scratch, st.rollout_model = 0, ep.kin_scratch.data_ptr(), 7   # only read with rollouts
    step()
    torch.cuda.synchronize()
    fab = Fabrics(R, device=0)
    d = torch.from_numpy(to_soa(rec)).to("cuda:0")
    with pytest.raises(MrfError):
        fab.rollout_cart_all_dev(d, torch.zeros((16, 10, 1, B), dtype=torch.float64, device="cuda:0"), 3)
    with pytest.raises(MrfError):
        fab.rollout_cart_all_dev(d[:, :1].contiguous(), None, 3)
    fab.close()
