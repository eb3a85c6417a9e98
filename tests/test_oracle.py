"""CPU tests of the oracle itself (no GPU): O2 (closed-form C) against the golden vectors made by O1 (autodiff,
fabrics-structured), FK known answers derived from the reference's constants, and the deadlock restatement against
golden sequences produced by the reference's own class."""
import os

import numpy as np
import pytest

from oracle import o2
from oracle.deadlock_ref import DeadlockOracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gold(built):
    return np.load(os.path.join(GOLD, "fabric_golden.npz"))


def test_fk_known_answers(built):
    """SURVEY Appendix B.2: at pos0 the hand sits at the reference's start goals (parameters_manipulators.py:93,126-128)
    -- validates chain constants, mount convention and that sub-goal 0 is expressed in the world frame."""
    pos0 = np.array([1.125, 0.19, 0.12, -1.66, 0.0, 1.88, np.pi / 4])
    cfg = o2.default_config(2)
    x0, *_ = o2.kinematics(cfg, 0, pos0, np.zeros(7))
    x1, *_ = o2.kinematics(cfg, 1, pos0, np.zeros(7))
    assert np.allclose(x0[2], [0.025732, 0.053847, 1.293313], atol=1e-6)
    assert np.allclose(x0[7], [0.204352, 0.589084, 1.147689], atol=1e-6)
    assert np.allclose(x1[7], [0.795648, -0.589084, 1.147689], atol=1e-6)
    assert np.linalg.norm(x0[7] - [0.2, 0.6, 1.15]) < 0.012
    assert np.linalg.norm(x1[7] - [0.8, -0.6, 1.15]) < 0.012
    assert np.array_equal(x0[0], x0[1]) and np.array_equal(x0[4], x0[5])     # link1==link2, link5==link6 origins
    R = o2.ROT_PANDA
    assert np.allclose(R @ (x0[7] - x0[6]), [0.106920, 0.003952, -0.001209], atol=1e-6)   # ~ x_goal_1


def test_o2_actions_match_o1_golden(gold):
    for c in range(int(gold["n_act"])):
        p = f"act{c}_"
        cfg = o2.default_config(3, mode=int(gold[p + "mode"]), has_collision_links=0 if int(gold[p + "grasp"]) else 1)
        obst = gold[p + "obst"]
        a, d = o2.action(cfg, int(gold[p + "robot"]), gold[p + "rec"], obst[:, 0:3], obst[:, 3:6], obst[:, 6:9],
                         obst[:, 9], want_diag=True)
        ref = gold[p + "action"]
        assert np.abs(a - ref).max() <= 1e-11 * max(1.0, np.abs(ref).max()), c
        for k in ("M_g", "f_g", "fe_g", "M_f", "f_f", "qdd"):
            assert np.abs(d[k] - gold[p + k]).max() <= 1e-11 * max(1.0, np.abs(gold[p + k]).max()), (c, k)


def test_o2_kinematics_match_o1_golden(gold):
    cfg = o2.default_config(3)
    rec = gold["kin_rec"]
    x, v, c, _ = o2.kinematics(cfg, int(gold["kin_robot"]), rec[0:7], rec[7:14])
    assert np.abs(x - gold["kin_xva"][:, 0]).max() < 1e-14
    assert np.abs(v - gold["kin_xva"][:, 1]).max() < 1e-14
    assert np.abs(-c - gold["kin_xva"][:, 2]).max() < 1e-13       # published a = Jdot_sign(-1) * d(J qd)/dq qd


def test_o2_rollouts_match_o1_golden(gold):
    cfg = o2.default_config(2)
    N = int(gold["ro_N"])
    qN, qdN, avg, _ = o2.rollout_jointspace(cfg, gold["ro_rec"], N)
    assert np.abs(qN - gold["ro_qN"]).max() < 1e-12
    assert np.abs(qdN - gold["ro_qdN"]).max() < 1e-11
    assert np.abs(avg - gold["ro_avg"]).max() < 1e-11
    obst = gold["cart_obst"]
    cq, cqd, cavg = o2.rollout_cartesian(cfg, 0, gold["cart_rec"], obst[:, 0:3], obst[:, 3:6], obst[:, 9], 2)
    assert np.abs(cq - gold["cart_qN"]).max() < 1e-12
    assert np.abs(cqd - gold["cart_qdN"]).max() < 1e-11
    assert abs(cavg - float(gold["cart_avg"])) < 1e-11


def test_o2_three_robot_rollout_matches_o1_golden(gold):
    """3 Pandas, unequal sphere radii, dynamic and static (STATIC_OR_DYN_FABRICS = 0) fabrics."""
    N = int(gold["ro3_N"])
    for sd in (1, 0):
        cfg = o2.default_config(3, static_or_dyn=sd)
        for r in range(3):
            for l in range(8):
                cfg.r_robots[r][l] = float(gold["ro3_rr"][r][l])
        qN, qdN, avg, _ = o2.rollout_jointspace(cfg, gold["ro3_rec"], N)
        assert np.abs(qN - gold[f"ro3_sd{sd}_qN"]).max() < 1e-12
        assert np.abs(qdN - gold[f"ro3_sd{sd}_qdN"]).max() < 1e-10
        assert np.abs(avg - gold[f"ro3_sd{sd}_avg"]).max() < 1e-10


def test_o1_live_matches_o2_small(built):
    """One live O1 evaluation (slow path, torch autodiff) so the generator of the golden file stays exercised."""
    from oracle import o1_fabrics as o1
    rng = np.random.default_rng(3)
    cfg = o2.default_config(2)
    rec = o2.make_record([0.9, 0.2, 0.1, -1.6, 0.2, 1.8, 0.5], rng.uniform(-0.5, 0.5, 7), [0.5, 0.1, 1.0], 2.0)
    obst = np.array([[0.6, 0.2, 1.2, 0.1, -0.2, 0.05, 0.3, 0.1, -0.2, 0.08]])
    pl = o1.make_panda_planner(o2.mount_of(cfg, 1), n_dyn=1)
    p = o2.record_to_params(rec)
    p.update(x_obst_dynamic_0=obst[0, 0:3], xdot_obst_dynamic_0=obst[0, 3:6], xddot_obst_dynamic_0=obst[0, 6:9],
             radius_obst_dynamic_0=obst[0, 9])
    a1, _ = pl.action_raw(rec[0:7], rec[7:14], p)
    a2 = o2.action(cfg, 1, rec, obst[:, 0:3], obst[:, 3:6], obst[:, 6:9], obst[:, 9])
    assert np.abs(a1 - a2).max() < 1e-11


def test_o1_matches_o2_link_subset_and_static_spheres(built):
    """Generic leaf set (SURVEY 8f rank 4): an arbitrary collision_links_nr subset (the reference's signature default is
    [5], example_pandas_Jointspace.py:64) and static spheres x_obst_i next to dynamic ones -- closed form (O2) against the
    autodiff derivation (O1)."""
    from oracle import o1_fabrics as o1
    rng = np.random.default_rng(5)
    rec = o2.make_record([0.9, 0.2, 0.1, -1.6, 0.2, 1.8, 0.5], rng.uniform(-0.5, 0.5, 7), [0.5, 0.1, 1.0], 2.0)
    dyn = np.array([[0.6, 0.2, 1.2, 0.1, -0.2, 0.05, 0.3, 0.1, -0.2, 0.08]])
    stat = np.array([[0.3, -0.4, 1.1, 0.07], [0.9, 0.5, 1.3, 0.1]])
    for links in ([5], [3, 6, 8], [1, 2, 4, 7]):
        cfg = o2.set_collision_links(o2.default_config(2), [[1, 2, 3, 4, 5, 6, 7, 8], links])
        pl = o1.make_panda_planner(o2.mount_of(cfg, 1), n_dyn=1, n_static=2,
                                   collision_links=[f"panda_link{l}" for l in links])
        r = rec.copy()
        r[o2.RB:o2.RB + 6] = [0.08 if (l in links) else 0.0 for l in range(3, 9)]
        p = o2.record_to_params(r)
        p.update(x_obst_dynamic_0=dyn[0, 0:3], xdot_obst_dynamic_0=dyn[0, 3:6], xddot_obst_dynamic_0=dyn[0, 6:9],
                 radius_obst_dynamic_0=dyn[0, 9], x_obst_0=stat[0, 0:3], radius_obst_0=stat[0, 3], x_obst_1=stat[1, 0:3],
                 radius_obst_1=stat[1, 3])
        a1, _ = pl.action_raw(r[0:7], r[7:14], p)
        # O2: static spheres are spheres at rest in the same list
        xo = np.vstack([stat[:, 0:3], dyn[:, 0:3]])
        vo = np.vstack([np.zeros((2, 3)), dyn[:, 3:6]])
        ao = np.vstack([np.zeros((2, 3)), dyn[:, 6:9]])
        ro = np.concatenate([stat[:, 3], dyn[:, 9]])
        a2 = o2.action(cfg, 1, r, xo, vo, ao, ro)
        assert np.abs(a1 - a2).max() < 1e-11, links
    full = o2.action(o2.default_config(2), 1, rec, xo, vo, ao, ro)
    assert np.abs(full - a2).max() > 1e-6                    # the subset really changes the action


def test_jdot_sign_and_eps_are_live_knobs(built):
    """The restatement assumptions (SURVEY A4/A7) are configuration, not constants: changing them changes the action."""
    rec = o2.make_record([0.9, 0.2, 0.1, -1.6, 0.2, 1.8, 0.5], [0.3, -0.2, 0.4, 0.1, -0.3, 0.2, 0.1], [0.5, 0.1, 1.0])
    obst = np.array([[0.6, 0.2, 1.2, 0.1, -0.2, 0.05, 0.0, 0.0, 0.0, 0.08]])
    base = o2.action(o2.default_config(2), 0, rec, obst[:, 0:3], obst[:, 3:6], obst[:, 6:9], obst[:, 9])
    plus = o2.action(o2.default_config(2, jdot_sign=1.0), 0, rec, obst[:, 0:3], obst[:, 3:6], obst[:, 6:9], obst[:, 9])
    assert np.abs(base - plus).max() > 1e-6


def test_deadlock_restatement_matches_reference_golden():
    g = np.load(os.path.join(GOLD, "deadlock_golden.npz"))
    raised = 0
    for c in range(int(g["n_cases"])):
        p = f"c{c}_"
        dl = DeadlockOracle(int(g[p + "R"]))
        tdo = 1000
        for t in range(len(g[p + "x"])):
            go, wo, tdo, flag = dl.step(g[p + "x"][t], g[p + "goals"][t], g[p + "weights"][t], int(g[p + "time_step"][t]),
                                        tdo, float(g[p + "avg"][t]), list(g[p + "states"][t]))
            raised += int(flag)
            assert np.array_equal(np.array(go), g[p + "goals_out"][t])
            assert np.array_equal(np.array(wo, dtype=float), g[p + "weights_out"][t])
            assert tdo == g[p + "tdo_out"][t]
    assert raised > 50


def test_deadlock_restatement_point_mass_branch_matches_reference_golden():
    """dof[0] == 2 constants (deadlock_prevention.py:12-19), sequences produced by the reference's own class."""
    g = np.load(os.path.join(GOLD, "deadlock_point_golden.npz"))
    raised = 0
    for c in range(int(g["n_cases"])):
        p = f"c{c}_"
        dl = DeadlockOracle(int(g[p + "R"]), point=True)
        tdo = 1000
        for t in range(len(g[p + "x"])):
            go, wo, tdo, flag = dl.step(g[p + "x"][t], g[p + "goals"][t], g[p + "weights"][t], int(g[p + "time_step"][t]),
                                        tdo, float(g[p + "avg"][t]), list(g[p + "states"][t]))
            raised += int(flag)
            assert np.array_equal(np.array(go), g[p + "goals_out"][t])
            assert np.array_equal(np.array(wo, dtype=float), g[p + "weights_out"][t])
            assert tdo == g[p + "tdo_out"][t]
    assert raised > 50


def test_sphere_offsets_and_sphere_kinematics(built):
    """Row 4 of the scope table: collision spheres with per-link offsets (create_simulation_manipulators.py:188-245,
    utils.py:87-119).  The package's offset table equals the oracle's restatement of the placement rule, and the
    closed-form sphere kinematics (O2) equal the autodiff ones (O1)."""
    from multi_robot_fabrics_b200.spheres import sphere_offsets
    from oracle import o1_fabrics as o1
    for n in (1, 2, 4, 5):
        assert np.array_equal(sphere_offsets(n), o2.sphere_offsets_ref(n))
    off4 = sphere_offsets(4)
    assert np.allclose(off4[0, :, 2], [-0.333, -0.24975, -0.1665, -0.08325])        # linear link: starts one length below
    assert np.allclose(off4[1, :, 2], [-0.1, -0.05, 0.0, 0.05])                      # rotational link: half a length
    assert np.allclose(off4[7, 1], [0.03, 0.03, 0.0]) and np.allclose(off4[7, 2], [-0.03, -0.03, 0.0])
    assert np.allclose(off4[4, 2], [0.0, 0.02, -0.192]) and np.allclose(off4[4, 3], [0.0, 0.06, -0.096])
    cfg = o2.default_config(3)
    rng = np.random.default_rng(0)
    q, qd = rng.uniform(-1, 1, 7), rng.uniform(-1, 1, 7)
    q[3] = -1.5
    off = sphere_offsets(2)
    x, vo, vs = o2.spheres(cfg, 2, q, qd, off)
    xl, vl, _, _ = o2.kinematics(cfg, 2, q, qd)
    for l in (0, 1, 4, 7):
        for s in range(2):
            xx, vv = o1.sphere_kinematics(q, qd, o2.mount_of(cfg, 2), f"panda_link{l + 1}", off[l, s])
            assert np.abs(xx - x[l * 2 + s]).max() < 1e-14 and np.abs(vv - vs[l * 2 + s]).max() < 1e-14
            assert np.array_equal(vo[l * 2 + s], vl[l])
    x1, _, _ = o2.spheres(cfg, 2, q, qd, np.zeros((8, 1, 3)))
    assert np.abs(x1 - xl).max() < 1e-15                                             # zero offsets = link origins


def test_point_mass_o2_matches_o1_golden(gold):
    """BASELINE config C1 (4 point masses): closed-form O2 against the O1 golden actions, static and dynamic variants
    (examples/example_pointmasses_static.py:191-199, examples/example_pointmasses_dynamic.py:192-212)."""
    cfg = o2.default_config(2)
    pos, vel, goals, obst = gold["pm_pos"], gold["pm_vel"], gold["pm_goals"], gold["pm_obst"]
    for i in range(4):
        others = [j for j in range(4) if j != i]
        a = o2.point_action(cfg, pos[i], vel[i], goals[i], 1.0, 0.2, np.concatenate([obst, pos[others]]), [1.0] * 6 + [0.2] * 3)
        assert np.abs(a - gold["pm_static"][i]).max() < 1e-12
        a = o2.point_action(cfg, pos[i], vel[i], goals[i], 1.0, 0.2, obst, [1.0] * 6, pos[others][:, 0:2],
                            vel[others][:, 0:2], np.zeros((3, 2)), [0.2] * 3)
        assert np.abs(a - gold["pm_dyn"][i]).max() < 1e-12


def test_fsm_restatement_matches_reference_golden():
    """SURVEY 8f rank 3: the state-machine restatement replays sequences produced by the reference's own class."""
    from oracle.fsm_ref import FsmOracle
    g = np.load(os.path.join(GOLD, "fsm_golden.npz"))
    seen = set()
    for c in range(int(g["n_cases"])):
        p = f"c{c}_"
        o = FsmOracle(g[p + "start"], int(g[p + "nr_blocks"]))
        for t in range(len(g[p + "x"])):
            st = o.step(g[p + "x"][t], g[p + "qg"][t], g[p + "gb"][t])
            seen.add(st)
            assert st == g[p + "state"][t] and np.array_equal(o.goal, g[p + "goal"][t]) and o.weight == g[p + "weight"][t]
            assert np.array_equal(o.gripper_action(g[p + "qg"][t]), g[p + "grip"][t])
    assert seen == {0, 1, 2, 3, 4, 5, 10, 12}


def test_assumption_knobs_agree_between_o1_and_o2(built):
    """The recalled fabrics internals (SURVEY A4/A7/A11) are knobs in every implementation.  With the alternative
    settings (Jdot sign +1, ExecutionLagrangian 0.5 qd.qd, eps 1e-5) the autodiff oracle and the closed form still agree,
    so if a real fabrics install ever shows a different convention, flipping the knob restores parity."""
    from oracle import o1_fabrics as o1
    rec = o2.make_record([0.9, 0.2, 0.1, -1.6, 0.2, 1.8, 0.5], [0.3, -0.2, 0.4, 0.1, -0.3, 0.2, 0.1], [0.5, 0.1, 1.0])
    obst = np.array([[0.6, 0.2, 1.2, 0.1, -0.2, 0.05, 0.3, 0.1, -0.2, 0.08], [0.2, -0.3, 1.3, 0.0, 0.1, 0.0, 0.0, 0.0, 0.0, 0.1]])
    kn = dict(jdot_sign=1.0, exec_scale=0.5, eps=1e-5)
    cfg = o2.default_config(2, **kn)
    pl = o1.make_panda_planner(o2.mount_of(cfg, 0), n_dyn=2, config=o1.panda_config(jdot_sign=1.0, exec_energy_scale=0.5, eps=1e-5))
    p = o2.record_to_params(rec)
    for i in range(2):
        p.update({f"x_obst_dynamic_{i}": obst[i, 0:3], f"xdot_obst_dynamic_{i}": obst[i, 3:6],
                  f"xddot_obst_dynamic_{i}": obst[i, 6:9], f"radius_obst_dynamic_{i}": obst[i, 9]})
    a1, _ = pl.action_raw(rec[0:7], rec[7:14], p)
    a2 = o2.action(cfg, 0, rec, obst[:, 0:3], obst[:, 3:6], obst[:, 6:9], obst[:, 9])
    assert np.abs(a1 - a2).max() < 1e-11
    base = o2.action(o2.default_config(2), 0, rec, obst[:, 0:3], obst[:, 3:6], obst[:, 6:9], obst[:, 9])
    assert np.abs(a2 - base).max() > 1e-6


def test_pick_and_place_cpu_loop_visits_the_protocol(built):
    """The CPU restatement of the pick-and-place control loop (the checker of the device control step) really grasps and
    releases a block: states leave 1, the gripper closes and re-opens, at least one block is counted."""
    from helpers import oracle_pick_and_place
    import multi_robot_fabrics_b200 as m
    R, nb = 2, 1
    rng = np.random.default_rng(9)
    rec = m.scenarios.generate(4, R, seed=91)
    rec[:, :, 7:14] = 0.0
    cfg = o2.default_config(R)
    b = 3
    start = np.array([o2.kinematics(cfg, r, rec[b, r, 0:7], rec[b, r, 7:14])[0][7] for r in range(R)])
    offs = rng.uniform(-0.06, 0.06, (4, R, 2))                       # blocks a few centimetres from the hands
    blocks = np.zeros((nb, R, 3))
    for r in range(R):
        blocks[0, r] = start[r] + np.array([offs[b, r, 0], offs[b, r, 1], -0.16])
    q, states, picked, n_flags, done_at, q_grip = oracle_pick_and_place(rec[b], blocks, start, 420, 3, estimate=True)
    assert np.isfinite(q).all() and picked.sum() >= 1 and 10 in states
