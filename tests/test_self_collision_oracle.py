"""Self-collision leaves: the kernels' closed form against autodiff (oracle O1), on the CPU."""
import numpy as np
import pytest
import torch

from oracle import o1_fabrics as o1
from oracle import o2
import self_collision_ref as sc

PAIRS = [(9, 2), (8, 3), (7, 4), (9, 1)]
LEAVES = [None, dict(k_geometry=-0.3, p_geometry=3, gate_geometry=0, k_finsler=0.05, p_finsler=4, gate_finsler=1)]


def _dist(q, mount, a, b):
    t = torch.as_tensor(q)
    pa = o1.panda_fk(t, mount, sc.LINK_NAMES[a]).numpy()
    pb = o1.panda_fk(t, mount, sc.LINK_NAMES[b]).numpy()
    return float(np.linalg.norm(pa - pb))


def _case(rng, R, robot, qd_kind):
    ocfg = o2.default_config(R)
    mount = o2.mount_of(ocfg, robot)
    lim = np.array(o1.PANDA_LIMITS)
    q = rng.uniform(lim[:, 0] + 0.3, lim[:, 1] - 0.3)
    qd = {"zero": np.zeros(7), "rand": rng.uniform(-0.6, 0.6, 7)}[qd_kind]
    # x = 0.3 for the first pair (close approach), 0.8 .. 2 for the others
    rho = [_dist(q, mount, *PAIRS[0]) / 1.3] + [_dist(q, mount, a, b) / rng.uniform(1.8, 3.0) for a, b in PAIRS[1:]]
    return ocfg, mount, q, qd, rho


@pytest.mark.parametrize("leaf", LEAVES, ids=["A13", "custom"])
@pytest.mark.parametrize("R,robot", [(2, 1), (3, 2)])
@pytest.mark.parametrize("qd_kind", ["zero", "rand"])
def test_closed_form_matches_autodiff(leaf, R, robot, qd_kind):
    rng = np.random.default_rng(7 + R + len(qd_kind))
    for _ in range(3):
        ocfg, mount, q, qd, rho = _case(rng, R, robot, qd_kind)
        Ma, fa, fea = sc.o1_pair_terms(q, qd, mount, PAIRS, rho, leaf)
        Mc, fc, fec = sc.closed_pair_terms(q, qd, mount, PAIRS, rho, leaf)
        for got, ref in ((Mc, Ma), (fc, fa), (fec, fea)):
            scale = max(np.abs(ref).max(), 1e-300)
            assert np.abs(got - ref).max() <= 1e-11 * scale + 1e-300


def test_sign_gate_both_directions():
    """xdot of both signs occurs among the pairs of the random cases (the gate is exercised on each side)."""
    rng = np.random.default_rng(3)
    signs = set()
    for _ in range(6):
        ocfg, mount, q, qd, rho = _case(rng, 2, 1, "rand")
        for a, b in PAIRS:
            x, v, _, _ = o1.link_kinematics(q, qd, mount, sc.LINK_NAMES[a])
            y, w, _, _ = o1.link_kinematics(q, qd, mount, sc.LINK_NAMES[b])
            signs.add(np.sign((x - y) @ (v - w)))
    assert {-1.0, 1.0} <= signs


@pytest.mark.parametrize("leaf", LEAVES, ids=["A13", "custom"])
def test_action_o1_vs_o2(leaf):
    """The whole action with pairs: O1 (autodiff planner and leaves) against O2 (closed form) to 1e-11."""
    rng = np.random.default_rng(11)
    for R, robot in ((2, 0), (3, 1)):
        ocfg, mount, q, qd, rho = _case(rng, R, robot, "rand")
        rec = o2.make_record(q, qd, x_goal_0=(0.5, 0.1 + robot * 0.2, 1.0))
        _, d2 = o2.action(ocfg, robot, rec, np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 3)), np.zeros(0), want_diag=True)
        a2 = sc.action_with_pairs(d2, rec, mount, PAIRS, rho, leaf, terms=sc.closed_pair_terms)
        pl = o1.make_panda_planner(mount, n_dyn=0)
        _, d1 = pl.action_raw(q, qd, o2.record_to_params(rec))
        a1 = sc.action_with_pairs(d1, rec, mount, PAIRS, rho, leaf, terms=sc.o1_pair_terms)
        assert np.abs(a1 - a2).max() <= 1e-11 * np.abs(a1).max()


def test_finish_action_reproduces_o2():
    """With no pairs, repeating the solve and damper on O2's diagnostics gives O2's own action."""
    rng = np.random.default_rng(5)
    ocfg, mount, q, qd, _ = _case(rng, 2, 1, "rand")
    rec = o2.make_record(q, qd, x_goal_0=(0.5, 0.3, 1.0))
    z = np.zeros((0, 3))
    out, d2 = o2.action(ocfg, 1, rec, z, z, z, np.zeros(0), want_diag=True)
    a = sc.action_with_pairs(d2, rec, mount, [], [])
    assert np.abs(a - out).max() <= 1e-12 * np.abs(out).max()


def test_coupled_rollout_without_pairs_is_o2():
    """The step loop the GPU tests replay with pairs gives O2's own coupled rollout when there are none."""
    import multi_robot_fabrics_b200 as m
    for R in (2, 3):
        rec = m.scenarios.generate(2, R, seed=40 + R)
        ocfg = o2.default_config(R)
        qN, qdN, _, _ = o2.rollout_jointspace(ocfg, rec, 4)
        for b in range(2):
            q1, qd1 = sc.coupled_rollout(ocfg, rec[b], 4, [], [])
            assert np.abs(qd1 - qdN[b]).max() <= 1e-12 * np.abs(qdN[b]).max()
            assert np.abs(q1 - qN[b]).max() <= 1e-12 * np.abs(qN[b]).max()


def test_closed_form_on_o2_kinematics():
    """The closed form fed with O2's point kinematics (what the CPU loops use) equals the autodiff terms."""
    rng = np.random.default_rng(21)
    for R, robot in ((2, 0), (3, 2)):
        ocfg, mount, q, qd, rho = _case(rng, R, robot, "rand")
        Ma, fa, fea = sc.o1_pair_terms(q, qd, mount, PAIRS, rho)
        Mc, fc, fec = sc.closed_pair_terms(q, qd, mount, PAIRS, rho, kin_of=sc.o2_kin(ocfg, robot))
        for got, ref in ((Mc, Ma), (fc, fa), (fec, fea)):
            assert np.abs(got - ref).max() <= 1e-11 * np.abs(ref).max()


@pytest.mark.parametrize("R", [2, 3])
def test_coupled_rollout_o1_vs_o2_with_pairs(R):
    """Short coupled rollout with pairs: O1 (autodiff planner, leaves and kinematics) against O2 + closed form."""
    import multi_robot_fabrics_b200 as m
    rec = m.scenarios.generate(1, R, seed=60 + R)[0]
    ocfg = o2.default_config(R)
    pairs = [PAIRS[:2], PAIRS[2:], PAIRS[1:3]][:R]
    rho = [[0.16] * len(p) for p in pairs]
    q2, qd2 = sc.coupled_rollout(ocfg, rec, 3, pairs, rho)
    q1, qd1 = sc.o1_coupled_rollout(ocfg, rec, 3, pairs, rho)
    assert np.abs(qd1 - qd2).max() <= 1e-11 * np.abs(qd1).max()
    assert np.abs(q1 - q2).max() <= 1e-11 * np.abs(q1).max()


def test_cartesian_rollout_o1_vs_o2_with_pairs():
    import multi_robot_fabrics_b200 as m
    from helpers import random_obstacles
    rec = m.scenarios.generate(1, 2, seed=71, weight_goal_1=20.0)
    obst = random_obstacles(np.random.default_rng(1), 1, 1, 3, rec[:, :1])[0, 0]
    obst[:, 6:9] = 0.0
    ocfg = o2.default_config(2)
    for leaf in LEAVES:
        a = sc.cartesian_rollout(ocfg, 0, rec[0, 0], obst, 4, PAIRS, [0.16] * 4, leaf)
        b = sc.cartesian_rollout(ocfg, 0, rec[0, 0], obst, 4, PAIRS, [0.16] * 4, leaf, use_o1=True)
        assert np.abs(a - b).max() <= 1e-11 * np.abs(b).max()


def test_dropin_pair_dict():
    """fabrics' dict form: names to link numbers, each unordered pair once, coincident pairs skipped with a warning."""
    from multi_robot_fabrics_b200.planner import self_collision_pair_list
    from multi_robot_fabrics_b200._lib import MrfError
    with pytest.warns(UserWarning):
        got = self_collision_pair_list({"panda_hand": ["panda_link2", "panda_link8"], "panda_link5": ["panda_link6"],
                                        "panda_link2": ["panda_hand"], "panda_link7": ["panda_link4"]})
    assert got == [(9, 2), (7, 4)]
    with pytest.raises(MrfError):
        self_collision_pair_list({"panda_link0": ["panda_link4"]})
