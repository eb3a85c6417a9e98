"""CPU tests of the point-mass scenario generator (scenarios.point_masses) that feeds episodes.BatchedPointEpisodes."""
import os

import numpy as np

import multi_robot_fabrics_b200 as m

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_point_masses_without_jitter_is_the_example():
    """jitter = 0 reproduces the scene tests/golden/make_fabric_golden.py stages for config C1 (stored in its output)."""
    g = np.load(os.path.join(GOLD, "fabric_golden.npz"))
    q0, goals, scene = m.scenarios.point_masses(5, seed=3)
    assert q0.shape == (5, 4, 3) and goals.shape == (5, 4, 2) and scene.shape == (5, 6, 4)
    for b in range(5):
        assert np.array_equal(q0[b], g["pm_pos"])
        assert np.array_equal(goals[b], g["pm_goals"])
        assert np.array_equal(scene[b, :, 0:3], g["pm_obst"])
    assert (scene[:, :, 3] == 1.0).all() and m.scenarios.POINT_RADIUS == 0.2


def test_point_masses_jitter_is_seeded_and_contact_free():
    a = m.scenarios.point_masses(500, seed=11, jitter=0.5)
    b = m.scenarios.point_masses(500, seed=11, jitter=0.5)
    c = m.scenarios.point_masses(500, seed=12, jitter=0.5)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert not np.array_equal(a[0], c[0])
    q0, goals, _ = a
    assert (m.scenarios.point_start_clearance(q0) > 0).all()
    assert (q0[:, :, 2] == 0).all()
    d0, dg = q0[:, :, 0:2] - m.scenarios.POINT_STARTS[:, 0:2], goals - m.scenarios.POINT_GOALS
    assert np.abs(d0).max() <= 0.5 and np.abs(dg).max() <= 0.5
    assert np.abs(d0).max() > 0.4 and np.abs(dg).max() > 0.4        # the offsets do span the interval


def test_point_masses_reach_is_seeded_and_solvable():
    """The solvable variant keeps point_masses' starts and scene; every goal lies 0.5 from its start, clear of the scene
    spheres and of the other goals by more than the margin."""
    q0, goals, scene = m.scenarios.point_masses_reach(300, seed=4)
    a = m.scenarios.point_masses(300, seed=4, jitter=0.3)
    assert np.array_equal(q0, a[0]) and np.array_equal(scene, a[2])
    assert np.array_equal(goals, m.scenarios.point_masses_reach(300, seed=4)[1])
    assert np.allclose(np.linalg.norm(goals - q0[:, :, 0:2], axis=-1), 0.5)
    gq = np.concatenate([goals, np.zeros((300, 4, 1))], axis=-1)
    assert (m.scenarios.point_start_clearance(gq) > 0.1).all()
