"""Host-pointer entries against the device-pointer entries, bit for bit.

The `_host` entries only stage: they move the caller's array-of-records arrays [B][A][F] to the kernels' layout
[F][A][B] and the results back.  So every output must equal what the device entry returns on the same inputs in
device layout, bitwise (compared through integer views, so that NaN compares equal), for every robot count and for
batches that are not multiples of the 32-wide staging tile.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from multi_robot_fabrics_b200._lib import check, hptr, lib
from multi_robot_fabrics_b200.api import Fabrics

from helpers import random_obstacles

TORCH = {"f64": "float64", "f32": "float32"}


@pytest.fixture(scope="module")
def fabs(built):
    d = {}
    yield d
    for f in d.values():
        f.close()


def _fourth_mount(fn):
    """Run fn with the fourth arm mounted away from the first one (by default both share a base)."""
    from multi_robot_fabrics_b200 import scenarios as sc
    old = sc.MOUNT_XYZ[3].copy()
    sc.MOUNT_XYZ[3] = [0.3, -0.6, 0.65]
    try:
        return fn(sc)
    finally:
        sc.MOUNT_XYZ[3] = old


def records(B, R, seed, **kw):
    return _fourth_mount(lambda sc: sc.generate(B, R, seed=seed, **kw))


def get_fab(fabs, R, **kw):
    key = (R, tuple(sorted(kw.items())))
    if key not in fabs:
        mounts = _fourth_mount(lambda sc: [sc.mount_matrix(r) for r in range(R)])
        fabs[key] = Fabrics(R, device=0, mount=mounts, **kw)
    return fabs[key]


def dev(a, perm, dtype):
    """Host array -> contiguous device tensor with its axes permuted to the device layout."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a).transpose(perm))).to("cuda:0", dtype=getattr(torch, TORCH[dtype]))


def assert_same_bits(host, d, perm, name):
    """host (numpy, host layout) equals the device tensor d permuted by `perm` into host layout, bit for bit."""
    import torch
    torch.cuda.synchronize()
    got = np.ascontiguousarray(d.permute(*perm).cpu().numpy())
    host = np.ascontiguousarray(host)
    assert got.shape == host.shape and got.dtype == host.dtype, name
    assert np.array_equal(host.view(np.uint8), got.view(np.uint8)), name


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("B", [1, 33, 37])
@pytest.mark.parametrize("R", [1, 2, 3, 4])
def test_rollout_host_equals_device(fabs, R, B, dtype):
    import torch
    N = 6
    rec = records(B, R, 300 + 10 * R + B)
    fab = get_fab(fabs, R, estimate_goal=1 if R > 1 else 0)
    host = fab.rollout_host(rec, N, dtype=dtype, trajectories=True)
    d_rec = dev(rec, (2, 1, 0), dtype)
    t = lambda *shape: torch.empty(shape, dtype=d_rec.dtype, device="cuda:0")
    xee, goal, qN, qdN = t(R, 3, B), t(3, B), t(R, N, 7, B), t(R, N, 7, B)
    avg = fab.rollout_dev(d_rec, N, x_ee=xee, goal_est=goal, qN=qN, qdN=qdN)
    assert_same_bits(host["avg_vel"], avg, (1, 0), "avg_vel")
    assert_same_bits(host["x_ee"], xee, (2, 0, 1), "x_ee")
    if R > 1:  # goal_est is only written when a robot's goal is estimated
        assert_same_bits(host["goal_est"], goal, (1, 0), "goal_est")
    assert_same_bits(host["qN"], qN, (3, 0, 1, 2), "qN")
    assert_same_bits(host["qdN"], qdN, (3, 0, 1, 2), "qdN")


@pytest.mark.parametrize("dtype", ["f64", "f32"])
def test_pipelined_rollout_host_equals_device(fabs, dtype):
    """A pageable batch of 8193 scenarios without trajectories takes the chunked pipeline (ragged last chunk)."""
    import torch
    R, N, B = 3, 5, 8193
    rec = np.tile(records(1024, R, 331), (9, 1, 1))[:B]
    rec[:, 0, 17] += np.arange(B) % 7 * 1e-3
    fab = get_fab(fabs, R, estimate_goal=1)
    host = fab.rollout_host(rec, N, dtype=dtype)
    d_rec = dev(rec, (2, 1, 0), dtype)
    xee = torch.empty((R, 3, B), dtype=d_rec.dtype, device="cuda:0")
    goal = torch.empty((3, B), dtype=d_rec.dtype, device="cuda:0")
    avg = fab.rollout_dev(d_rec, N, x_ee=xee, goal_est=goal)
    assert_same_bits(host["avg_vel"], avg, (1, 0), "avg_vel")
    assert_same_bits(host["x_ee"], xee, (2, 0, 1), "x_ee")
    assert_same_bits(host["goal_est"], goal, (1, 0), "goal_est")


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("R,n_rob,robot_first,S,B", [(3, 2, 1, 7, 37), (3, 3, 0, 0, 33), (2, 1, 1, 5, 1), (4, 4, 0, 3, 40),
                                                     (2, 2, 0, 0, 1)])
def test_action_host_equals_device(fabs, R, n_rob, robot_first, S, B, dtype):
    rng = np.random.default_rng(R + 10 * n_rob + S)
    rec = records(B, R, 340 + S, weight_goal_1=20.0)[:, robot_first:robot_first + n_rob]
    obst = random_obstacles(rng, B, n_rob, S, rec, robot_first=robot_first)
    fab = get_fab(fabs, R)
    act = fab.action_host(rec, obst if S else None, robot_first=robot_first, dtype=dtype)
    d_act = fab.action_dev(dev(rec, (2, 1, 0), dtype), dev(obst, (2, 3, 1, 0), dtype) if S else None,
                           robot_first=robot_first)
    assert_same_bits(act, d_act, (2, 1, 0), "action")


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("S,B", [(0, 33), (16, 37)])
def test_rollout_cart_host_equals_device(fabs, S, B, dtype):
    import torch
    R, N = 2, 7
    rng = np.random.default_rng(350 + S)
    rec = records(B, R, 351, weight_goal_1=20.0)
    fab = get_fab(fabs, R)
    for robot in range(R):
        obst = random_obstacles(rng, B, 1, S, rec[:, robot:robot + 1], robot_first=robot)[:, 0]
        avg, qN, qdN = fab.rollout_cart_host(robot, rec[:, robot], obst, N, dtype=dtype)
        d_rec = dev(rec[:, robot], (1, 0), dtype)
        d_qN = torch.empty((N, 7, B), dtype=d_rec.dtype, device="cuda:0")
        d_qdN = torch.empty_like(d_qN)
        d_avg = fab.rollout_cart_dev(robot, d_rec, dev(obst, (1, 2, 0), dtype) if S else None, N, qN=d_qN, qdN=d_qdN)
        assert_same_bits(avg, d_avg, (0,), "avg_vel")
        assert_same_bits(qN, d_qN, (2, 0, 1), "qN")
        assert_same_bits(qdN, d_qdN, (2, 0, 1), "qdN")


@pytest.mark.parametrize("B", [1, 37])
@pytest.mark.parametrize("R", [1, 2, 3, 4])
def test_kinematics_host_equals_device(fabs, R, B):
    rec = records(B, R, 360 + R)
    fab = get_fab(fabs, R)
    x, v, a = fab.kinematics_host(rec[..., 0:7], rec[..., 7:14])
    dx, dv, da = fab.kinematics_dev(dev(rec[..., 0:7], (2, 1, 0), "f64"), dev(rec[..., 7:14], (2, 1, 0), "f64"))
    for name, h, d in (("x", x, dx), ("v", v, dv), ("a", a, da)):
        assert_same_bits(h, d, (3, 2, 0, 1), name)


@pytest.mark.parametrize("Ss,Sd,B", [(0, 0, 33), (3, 0, 37), (0, 2, 1), (4, 3, 70)])
def test_point_action_host_equals_device(fabs, Ss, Sd, B):
    rng = np.random.default_rng(370 + Ss + 10 * Sd)
    rec = np.zeros((B, 10))
    rec[:, 0:3] = rng.uniform(-2, 2, (B, 3))                 # q (x, y, theta)
    rec[:, 3:6] = rng.uniform(-0.5, 0.5, (B, 3))             # qdot
    rec[:, 6:8] = rng.uniform(-2, 2, (B, 2))                 # goal
    rec[:, 8], rec[:, 9] = 1.0, 0.2                          # goal weight, body radius
    stat = np.concatenate([rng.uniform(-3, 3, (B, Ss, 3)), rng.uniform(0.1, 0.5, (B, Ss, 1))], axis=2)
    dyn = np.concatenate([rng.uniform(-3, 3, (B, Sd, 2)), rng.uniform(-0.5, 0.5, (B, Sd, 4)),
                          rng.uniform(0.1, 0.5, (B, Sd, 1))], axis=2)
    fab = get_fab(fabs, 2)
    act = np.empty((B, 3))
    check(lib().mrf_point_action_host_f64(fab.handle.ptr, hptr(rec), Ss, hptr(stat) if Ss else None, Sd,
                                          hptr(dyn) if Sd else None, hptr(act), C.c_int64(B)), "mrf_point_action_host")
    d_act = fab.point_action_dev(dev(rec, (1, 0), "f64"), dev(stat, (1, 2, 0), "f64") if Ss else None,
                                 dev(dyn, (1, 2, 0), "f64") if Sd else None)
    assert_same_bits(act, d_act, (1, 0), "action")
