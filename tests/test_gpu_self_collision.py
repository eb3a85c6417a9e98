"""Self-collision pairs on the B200: executed action and coupled rollouts against the float64 oracle with the pair leaves,
host entries against device entries, clearing, argument checks and the entries that refuse pairs."""
import numpy as np
import pytest

import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200.api import Fabrics, to_soa
from multi_robot_fabrics_b200._lib import MrfError
from oracle import o2

import self_collision_ref as sc
from helpers import random_obstacles, rel_ps

pytestmark = pytest.mark.gpu
F64_RTOL = 1e-9
PAIRS = [[(9, 2), (8, 3)], [(7, 4), (9, 1), (8, 4)], [(9, 3)], [(7, 3), (9, 2)]]
LEAF2 = dict(k_geometry=-0.3, p_geometry=3, gate_geometry=0, k_finsler=0.05, p_finsler=4, gate_finsler=1)


def _rho(R):
    return [[0.16] * len(PAIRS[r]) for r in range(R)]


def _ref_actions(rec, obst, R, robot_first, leaf=None, **cfgkw):
    ocfg = o2.default_config(R, **cfgkw)
    B, n_rob = rec.shape[:2]
    out = np.full((B, n_rob, 7), np.nan)
    for b in range(B):
        for i in range(n_rob):
            r = robot_first + i
            o = obst[b, i]
            try:
                _, d = o2.action(ocfg, r, rec[b, i], o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9], want_diag=True)
            except FloatingPointError:
                continue
            out[b, i] = sc.action_with_pairs(d, rec[b, i], o2.mount_of(ocfg, r), PAIRS[r], _rho(4)[r], leaf,
                                             mode="vel" if ocfg.mode == 1 else "acc")
    return out


@pytest.mark.parametrize("R,robot_first,n_rob,S,kw", [(2, 0, 2, 8, {}), (3, 1, 2, 0, {}), (3, 2, 1, 4, {}),
                                                      (2, 0, 2, 4, dict(has_collision_links=0))])
@pytest.mark.parametrize("leaf", [None, LEAF2], ids=["A13", "custom"])
def test_action_matches_oracle(built, R, robot_first, n_rob, S, kw, leaf):
    B = 24
    rng = np.random.default_rng(R * 10 + S)
    rec = m.scenarios.generate(B, R, seed=31, weight_goal_1=20.0)[:, robot_first:robot_first + n_rob]
    obst = random_obstacles(rng, B, n_rob, S, rec, robot_first=robot_first)
    fab = Fabrics(R, device=0, **kw)
    try:
        fab.set_self_collision(PAIRS[:R], _rho(R), leaf)
        ref = _ref_actions(rec, obst, R, robot_first, leaf, **kw)
        ok = np.isfinite(ref).all(axis=(1, 2))
        assert ok.sum() > 0.8 * B
        act = fab.action_host(rec, obst if S else None, robot_first=robot_first, dtype="f64")
        assert rel_ps(act, ref, ok) < F64_RTOL
        act32 = fab.action_host(rec, obst if S else None, robot_first=robot_first, dtype="f32")
        assert np.abs(act32 - ref)[ok].max() < 2e-3
        # the pairs change the action: the leaves are really evaluated
        fab.set_self_collision(None, None)
        act0 = fab.action_host(rec, obst if S else None, robot_first=robot_first, dtype="f64")
        assert np.abs(act0 - act).max() > 1e-6
    finally:
        fab.close()


@pytest.mark.parametrize("R,B", [(1, 3), (2, 5), (3, 600), (4, 2)])
def test_coupled_rollout_matches_oracle(built, R, B):
    """Generic kernel at every batch size (B = 600 is above the cooperative kernel's threshold, the others below)."""
    import torch
    N = 6
    ocfg = o2.default_config(R)
    mounts = [o2.mount_of(ocfg, r) for r in range(R)]
    if R == 4:  # by default the fourth arm shares the first one's base: mount it apart, in the scenarios and both planners
        from multi_robot_fabrics_b200 import scenarios as scn
        old = scn.MOUNT_XYZ[3].copy()
        scn.MOUNT_XYZ[3] = [0.3, -0.6, 0.65]
        try:
            rec = scn.generate(B, R, seed=50 + R)
        finally:
            scn.MOUNT_XYZ[3] = old
        mounts[3][0:3, 3] = [0.3, -0.6, 0.65]
        for i, v in enumerate(mounts[3].reshape(16)):
            ocfg.mount[3][i] = v
    else:
        rec = m.scenarios.generate(B, R, seed=50 + R)
    fab = Fabrics(R, device=0, mount=mounts)
    try:
        fab.set_self_collision(PAIRS[:R], _rho(R))
        out = fab.rollout_host(rec, N, dtype="f64", trajectories=True)
        for b in sorted({0, B // 2, B - 1}):
            qN, qdN = sc.coupled_rollout(ocfg, rec[b], N, PAIRS[:R], _rho(R))
            e_qd = np.abs(out["qdN"][b] - qdN).max() / np.abs(qdN).max()
            e_q = np.abs(out["qN"][b] - qN).max() / np.abs(qN).max()
            assert e_qd < F64_RTOL and e_q < F64_RTOL, (b, e_qd, e_q)
        # the device entry, called with the same outputs, gives the host entry's bits
        d_rec = torch.from_numpy(to_soa(rec)).to("cuda:0")
        qdN_d = torch.empty((R, N, 7, B), dtype=torch.float64, device="cuda:0")
        xee = torch.empty((R, 3, B), dtype=torch.float64, device="cuda:0")
        ge = torch.empty((3, B), dtype=torch.float64, device="cuda:0")
        qN_d = torch.empty_like(qdN_d)
        avg = fab.rollout_dev(d_rec, N, x_ee=xee, goal_est=ge, qN=qN_d, qdN=qdN_d)
        assert np.array_equal(avg.cpu().numpy().T, out["avg_vel"], equal_nan=True)  # blown-up scenarios are NaN in both
        assert np.array_equal(np.moveaxis(qdN_d.cpu().numpy(), 3, 0), out["qdN"], equal_nan=True)
        # FP32 within the FP32 rollout tests' bound, on the scenarios that stay well conditioned (as oracle_rollout's mask)
        o32 = fab.rollout_host(rec, N, dtype="f32", trajectories=True)
        mx = np.abs(out["qdN"]).max(axis=(1, 2, 3))
        ok = np.isfinite(mx) & (mx < 3.0)
        assert ok.sum() >= 0.9 * B
        assert np.abs(o32["qdN"] - out["qdN"])[ok].max() < 2e-3
    finally:
        fab.close()


def test_cartesian_rollouts_match_oracle(built):
    """Cartesian rollout (one robot, spheres at constant velocity) with pairs: N steps of the action with the spheres
    moved, against the oracle's action with pairs."""
    B, N, S, R = 6, 5, 4, 2
    rng = np.random.default_rng(8)
    rec = m.scenarios.generate(B, R, seed=13, weight_goal_1=20.0)
    obst = random_obstacles(rng, B, 1, S, rec[:, :1])[:, 0]
    obst[..., 6:9] = 0.0
    fab = Fabrics(R, device=0)
    try:
        fab.set_self_collision(PAIRS[:R], _rho(R))
        _, _, qdN_c = fab.rollout_cart_host(0, rec[:, 0], obst, N, dtype="f64", trajectories=True)
        ocfg = o2.default_config(R)
        for b in range(B):
            cur = rec[b, 0].copy()
            xo = obst[b, :, 0:3].copy()
            for k in range(N):
                _, d = o2.action(ocfg, 0, cur, xo, obst[b, :, 3:6], obst[b, :, 6:9], obst[b, :, 9], want_diag=True)
                qd = sc.action_with_pairs(d, cur, o2.mount_of(ocfg, 0), PAIRS[0], _rho(R)[0])
                cur[7:14] = qd
                cur[0:7] = cur[0:7] + ocfg.dt * qd
                xo = xo + ocfg.dt * obst[b, :, 3:6]
                assert np.abs(qdN_c[b, k] - qd).max() / np.abs(qd).max() < F64_RTOL
    finally:
        fab.close()


def test_clearing_restores_the_plain_planner(built):
    R, B, N, S = 3, 40, 5, 4
    rng = np.random.default_rng(2)
    rec = m.scenarios.generate(B, R, seed=9)
    obst = random_obstacles(rng, B, R, S, rec)
    plain, fab = Fabrics(R, device=0), Fabrics(R, device=0)
    try:
        fab.set_self_collision(PAIRS[:R], _rho(R))
        fab.action_host(rec, obst)
        fab.set_self_collision([[], [], []], [[], [], []])
        for dt in ("f64", "f32"):
            assert np.array_equal(fab.action_host(rec, obst, dtype=dt), plain.action_host(rec, obst, dtype=dt))
            a, b = fab.rollout_host(rec, N, dtype=dt, trajectories=True), plain.rollout_host(rec, N, dtype=dt, trajectories=True)
            for k in a:
                assert np.array_equal(a[k], b[k]), k
    finally:
        plain.close()
        fab.close()


def test_setter_rejections_and_unsupported_entries(built):
    import torch
    fab = Fabrics(2, device=0)
    try:
        bad = [
            ([[(5, 6)]], [[0.1]]), ([[(8, 9)]], [[0.1]]), ([[(4, 4)]], [[0.1]]), ([[(1, 2)]], [[0.1]]),
            ([[(0, 4)]], [[0.1]]), ([[(3, 10)]], [[0.1]]), ([[(9, 3)]], [[0.0]]), ([[(9, 3)]], [[-1.0]]),
            ([[], [], [(9, 3)]], [[], [], [0.1]]),       # robot the handle does not have
            ([[(9, 3)] * 9], [[0.1] * 9]),               # more than MRF_MAX_SELF_PAIRS
        ]
        for pairs, rho in bad:
            with pytest.raises(MrfError):
                fab.set_self_collision(pairs, rho)
        for leaf in (dict(p_geometry=0), dict(p_finsler=9), dict(gate_geometry=2), dict(gate_finsler=-1),
                     dict(k_finsler=float("nan"))):
            with pytest.raises(MrfError):
                fab.set_self_collision([[(9, 3)]], [[0.1]], leaf)
        fab.set_self_collision([[(9, 3)], [(9, 2)]], [[0.1], [0.1]])
        rec = m.scenarios.generate(64, 2, seed=1)
        d_rec = torch.from_numpy(to_soa(rec)).to("cuda:0", dtype=torch.float32)
        risk = torch.empty((2, 64), dtype=torch.float32, device="cuda:0")
        with pytest.raises(MrfError, match="-5"):
            fab.rollout_dev(d_rec, 5, risk=risk)
        out = {k: np.empty(s, np.float32) for k, s in (("avg_vel", (64, 2)), ("x_ee", (64, 2, 3)), ("goal_est", (64, 3)))}
        with pytest.raises(MrfError, match="-5"):
            fab.rollout_host_submit(rec.astype(np.float32), 5, out)
    finally:
        fab.close()


def test_more_unsupported_entries(built):
    """Every entry that cannot evaluate the leaves refuses with MRF_EUNSUPPORTED (-5) while pairs are set."""
    import ctypes as C
    import torch
    from multi_robot_fabrics_b200._lib import lib
    R, B, N = 2, 64, 5
    fab = Fabrics(R, device=0)
    try:
        fab.set_self_collision([[(9, 3)], [(9, 2)]], [[0.16], [0.16]])
        rec = m.scenarios.generate(B, R, seed=2)
        d64 = torch.from_numpy(to_soa(rec)).to("cuda:0")
        with pytest.raises(MrfError, match="-5"):
            fab.rollout_dev(d64, N, risk=torch.empty((R, B), dtype=torch.float64, device="cuda:0"))
        h32 = rec.astype(np.float32)
        res = np.empty((R + 1, B), np.float32)
        with pytest.raises(MrfError, match="-5"):
            fab.rfcv_host_submit(h32, N, res)
        p = lambda a: C.c_void_p(a.ctypes.data)
        avg, xee, ge = np.empty((B, R), np.float32), np.empty((B, R, 3), np.float32), np.empty((B, 3), np.float32)
        shared = np.ascontiguousarray(h32[0])
        rc = lib().mrf_rollout_host_submit_compact_f32(fab.handle.ptr, p(np.ascontiguousarray(h32[:, :, :18])), p(shared), N,
                                                       p(avg), p(xee), p(ge), B)
        assert rc == -5
        rc = lib().mrf_rollout_host_submit_compact_f64(fab.handle.ptr, p(np.ascontiguousarray(rec[:, :, :18])),
                                                       p(np.ascontiguousarray(rec[0])), N, p(avg.astype(np.float64)),
                                                       p(xee.astype(np.float64)), p(ge.astype(np.float64)), B)
        assert rc == -5
        # mrf_rfcv_post_dev_f32 with a risk array: its FP64 guard re-roll has no pair loop
        d32 = torch.from_numpy(to_soa(rec)).to("cuda:0", dtype=torch.float32)
        f = lambda *s: torch.zeros(s, dtype=torch.float32, device="cuda:0")
        i = lambda *s: torch.zeros(s, dtype=torch.int32, device="cuda:0")
        work, x, g, av, risk = d32.clone(), f(R, 3, B), f(3, B), f(R, B), f(R, B)
        sm, ts, tdo, st_int, st_goal, flag, result = i(R, B), i(B), i(B), i(4 * B), f(3, B), i(B), f(R + 1, B)
        q = lambda t: C.c_void_p(t.data_ptr())
        rc = lib().mrf_rfcv_post_dev_f32(fab.handle.ptr, q(d32), N, q(x), q(work), q(g), q(av), q(risk), q(sm), q(ts), q(tdo),
                                         q(st_int), q(st_goal), q(flag), q(result), B, None, 0)
        assert rc == -5
    finally:
        fab.close()


def test_host_entries_equal_device_entries_with_pairs(built):
    """Action, Cartesian (one robot and all robots) and large page-locked rollouts: host entries give the device entries'
    bits with pairs set; page-locked records of a large batch take the staged path (no in-place read with pairs)."""
    import torch
    R, B, S, N = 3, 40, 4, 4
    rng = np.random.default_rng(4)
    rec = m.scenarios.generate(B, R, seed=19, weight_goal_1=20.0)
    obst = random_obstacles(rng, B, R, S, rec)
    fab = Fabrics(R, device=0)
    try:
        fab.set_self_collision(PAIRS[:R], _rho(R))
        for dt, tdt in (("f64", torch.float64), ("f32", torch.float32)):
            d_rec = torch.from_numpy(to_soa(rec)).to("cuda:0", dtype=tdt)
            d_obst = torch.from_numpy(np.ascontiguousarray(np.transpose(obst, (2, 3, 1, 0)))).to("cuda:0", dtype=tdt)
            a_dev = fab.action_dev(d_rec, d_obst).cpu().numpy()                            # (7,R,B)
            a_host = fab.action_host(rec, obst, dtype=dt)                                  # (B,R,7)
            assert np.array_equal(np.transpose(a_dev, (2, 1, 0)), a_host, equal_nan=True)
            qdN_all = torch.empty((R, N, 7, B), dtype=tdt, device="cuda:0")
            fab.rollout_cart_all_dev(d_rec, d_obst, N, qdN=qdN_all)
            for r in range(R):
                _, _, qdN_h = fab.rollout_cart_host(r, rec[:, r], obst[:, r], N, dtype=dt, trajectories=True)
                assert np.array_equal(np.moveaxis(qdN_all[r].cpu().numpy(), 2, 0), qdN_h, equal_nan=True), r
        Bl = 8192
        big = m.scenarios.generate(Bl, 2, seed=23)
        fab2 = Fabrics(2, device=0)
        try:
            fab2.set_self_collision(PAIRS[:2], _rho(2))
            pinned = torch.empty((Bl, 2, 44), dtype=torch.float32, pin_memory=True)
            pinned.copy_(torch.from_numpy(big))
            out = fab2.rollout_host(pinned.numpy(), N, dtype="f32")
            d = torch.from_numpy(to_soa(big)).to("cuda:0", dtype=torch.float32)
            xee = torch.empty((2, 3, Bl), dtype=torch.float32, device="cuda:0")
            ge = torch.empty((3, Bl), dtype=torch.float32, device="cuda:0")
            avg = fab2.rollout_dev(d, N, x_ee=xee, goal_est=ge)
            assert np.array_equal(avg.cpu().numpy().T, out["avg_vel"], equal_nan=True)
        finally:
            fab2.close()
    finally:
        fab.close()


@pytest.mark.parametrize("kw", [dict(), dict(estimate_goal=True)], ids=["RF", "RF-CV"])
def test_batched_episodes_with_pairs_match_cpu_loop(built, kw):
    """25 reach steps of BatchedEpisodes(self_collision_pairs=...) against the CPU loop with O2 and the pair leaves."""
    from multi_robot_fabrics_b200.episodes import BatchedEpisodes
    R, B, T, N = 2, 3, 25, 5
    rec = m.scenarios.generate(B, R, seed=81)
    pairs, rho = PAIRS[:R], _rho(R)
    ep = BatchedEpisodes(rec, n_horizon=N, dtype="f64", self_collision_pairs=pairs, self_collision_rho=rho, **kw).run(T)
    res = ep.results()
    for b in range(B):
        q, n_flags, done_at = sc.episode(rec[b], T, N, pairs, rho, estimate=kw.get("estimate_goal", False))
        assert np.abs(res["q"][b] - q).max() < 1e-7, b
        assert res["deadlock_steps"][b] == n_flags and res["steps_to_success"][b] == done_at


def test_pick_and_place_with_pairs_reaches_grasp_state(built):
    """Pick-and-place with pairs (grasp planner of state 2 included) against the CPU loop."""
    from multi_robot_fabrics_b200.episodes import BatchedEpisodes
    R, B, T, N, nb = 2, 2, 150, 3, 1
    rng = np.random.default_rng(9)
    rec = m.scenarios.generate(B, R, seed=91)
    rec[:, :, 7:14] = 0.0
    cfg = o2.default_config(R)
    start, blocks = np.zeros((B, R, 3)), np.zeros((B, nb, R, 3))
    for b in range(B):
        for r in range(R):
            start[b, r] = o2.kinematics(cfg, r, rec[b, r, 0:7], rec[b, r, 7:14])[0][7]
            blocks[b, 0, r] = start[b, r] + np.array([rng.uniform(-0.06, 0.06), rng.uniform(-0.06, 0.06), -0.16])
    pairs, rho = [[(9, 2), (7, 3)], [(9, 1)]], [[0.16, 0.16], [0.16]]
    ep = BatchedEpisodes(rec, n_horizon=N, dtype="f64", blocks=blocks, start_goal=start, self_collision_pairs=pairs,
                         self_collision_rho=rho).run(T)
    res = ep.results()
    seen_all = set()
    for b in range(B):
        q, states, picked, n_flags, done_at, q_grip, seen = sc.pick_and_place(rec[b], blocks[b], start[b], T, N, pairs, rho)
        seen_all |= seen
        assert np.array_equal(res["state"][b], states) and np.array_equal(res["blocks_picked"][b], picked), b
        assert res["steps_to_success"][b] == done_at and res["deadlock_steps"][b] == n_flags
        assert np.abs(res["q"][b] - q).max() < 1e-7
    assert 2 in seen_all            # the grasp planner ran with the pairs


def test_dropin_compute_action_with_pairs_matches_o1(built):
    """set_planner_panda(..., self_collision_pairs=fabrics' dict).compute_action(**kwargs) against O1 with the leaves;
    rho comes from radius_body_panda_links / radius_body_panda_hand, a missing radius raises."""
    import warnings as W
    from multi_robot_fabrics_b200 import planner as P
    from oracle import o1_fabrics as o1
    mount_param = {"mount_positions": [[0.0, 0.0, 0.0], [1.0, 0.0, 0.0]]}
    links = [1, 2, 3, 4, 5, 6, 7, 8]
    pairs_dict = {"panda_hand": ["panda_link2", "panda_link3"], "panda_link7": ["panda_link4"], "panda_link5": ["panda_link6"]}
    with W.catch_warnings(record=True) as caught:
        W.simplefilter("always")
        pl, _ = P.set_planner_panda(7, 0, 0, links, {}, mount_param, 0, self_collision_pairs=pairs_dict)
    assert any("coincide" in str(c.message) for c in caught)                  # (5, 6) skipped
    try:
        rng = np.random.default_rng(3)
        rec = m.scenarios.generate(6, 2, seed=33, weight_goal_1=20.0)[:, 0]
        radii = {str(l): 0.07 + 0.005 * l for l in range(1, 9)}
        o1pl = o1.make_panda_planner(pl.mount, n_dyn=0)
        for b in range(6):
            r = rec[b]
            kw = dict(q=r[0:7], qdot=r[7:14], x_goal_0=r[14:17], weight_goal_0=r[17], x_goal_1=r[18:21],
                      weight_goal_1=r[21], x_goal_2=r[22:23], weight_goal_2=r[23], angle_goal_1=r[24:33].reshape(3, 3),
                      constraint_0=r[33:37], radius_body_panda_links=radii, radius_body_panda_hand=0.09)
            act = pl.compute_action(**kw)
            rr = r.copy()
            rr[37:43] = [radii[str(l)] for l in range(3, 9)]
            _, d = o1pl.action_raw(r[0:7], r[7:14], o2.record_to_params(rr))
            pairs = [(9, 2), (9, 3), (7, 4)]
            rad = lambda l: 0.09 if l == 9 else radii[str(l)]
            ref = sc.action_with_pairs(d, rr, pl.mount, pairs, [rad(a) + rad(c) for a, c in pairs], terms=sc.o1_pair_terms)
            assert np.abs(act - ref).max() <= 1e-9 * np.abs(ref).max()
        assert pl.self_rho == [0.09 + radii["2"], 0.09 + radii["3"], radii["7"] + radii["4"]]
        kw.pop("radius_body_panda_hand")
        with pytest.raises(MrfError):
            pl.compute_action(**kw)
    finally:
        pl.fab.close()
