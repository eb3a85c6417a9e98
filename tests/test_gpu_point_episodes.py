"""GPU tests of the closed-loop point-mass episodes (episodes.BatchedPointEpisodes, mrf_point_episode_run_dev_*): the
control loops of examples/example_pointmasses_static.py and _dynamic.py, many control steps per kernel launch, against
the same loop run on the CPU with oracle O2's point-mass planner."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200._lib import MrfError, check, default_config, lib
from multi_robot_fabrics_b200.api import Fabrics
from multi_robot_fabrics_b200.episodes import BatchedPointEpisodes
from oracle import o2


def cpu_point_loop(q0, goals, scene, dynamic, T, qd0=None, radius=0.2, weight=1.0, epsilon=0.05, q_in=None):
    """CPU restatement of the point-mass control loop (include/mrf_b200.h, MrfPointEpisode) for ONE scenario:
    q0 (R,3), goals (R,2), scene (S,4).  q_in (R,3) perturbs the state the loop starts from (sensitivity).
    -> dict(traj (T,R,3), done_at, min_clear_robots, min_clear_scene, nonfinite_steps)"""
    cfg, dt = o2.default_config(2), float(default_config(1).dt)
    R = q0.shape[0]
    q = (q0 if q_in is None else q_in).astype(np.float64).copy()
    qd = np.zeros((R, 3)) if qd0 is None else qd0.astype(np.float64).copy()
    traj, done, mrr, msc, nbad = np.zeros((T, R, 3)), -1, np.inf, np.inf, 0
    for t in range(T):
        if done < 0 and all(np.sqrt((q[i, 0] - goals[i, 0]) ** 2 + (q[i, 1] - goals[i, 1]) ** 2) < epsilon for i in range(R)):
            done = t
        a, bad = np.zeros((R, 3)), False
        for i in range(R):
            oth = [j for j in range(R) if j != i]
            for j in oth:
                mrr = min(mrr, np.sqrt((q[i, 0] - q[j, 0]) ** 2 + (q[i, 1] - q[j, 1]) ** 2) - (radius + radius))
            for o in scene:
                msc = min(msc, np.sqrt((q[i, 0] - o[0]) ** 2 + (q[i, 1] - o[1]) ** 2 + (0.05 - o[2]) ** 2) - (o[3] + radius))
            if dynamic:
                ai = o2.point_action(cfg, q[i], qd[i], goals[i], weight, radius, scene[:, 0:3], scene[:, 3],
                                     q[oth, 0:2], qd[oth, 0:2], np.zeros((R - 1, 2)), [radius] * (R - 1))
            else:
                ai = o2.point_action(cfg, q[i], qd[i], goals[i], weight, radius, np.concatenate([scene[:, 0:3], q[oth]]),
                                     np.concatenate([scene[:, 3], [radius] * (R - 1)]))
            if not np.isfinite(ai).all():
                ai, bad = np.zeros(3), True
            a[i] = ai
        nbad += bad
        qd = qd + dt * a
        q = q + dt * qd
        traj[t] = q
    return dict(traj=traj, done_at=done, min_clear_robots=mrr, min_clear_scene=msc, nonfinite_steps=nbad)


def random_scenes(B, R, seed, half=4.0):
    """B scenarios of R point robots (radius 0.2) placed uniformly in [-half, half]^2 among the examples' 6 scene spheres,
    contact-free at the start, with random goals and velocities."""
    rng = np.random.default_rng(seed)
    q0 = np.zeros((B, R, 3))
    for b in range(B):
        while True:
            q = np.zeros((1, R, 3))
            q[0, :, 0:2] = rng.uniform(-half, half, (R, 2))
            if m.scenarios.point_start_clearance(q)[0] > 0.1:
                q0[b] = q[0]
                break
    goals = rng.uniform(-half, half, (B, R, 2))
    qd0 = np.zeros((B, R, 3))
    qd0[:, :, 0:2] = rng.uniform(-0.5, 0.5, (B, R, 2))
    scene = m.scenarios.point_masses(B)[2]
    return q0, goals, scene, qd0


def run(q0, goals, scene, dynamic, T, dtype="f64", chunks=None, **kw):
    ep = BatchedPointEpisodes(q0, goals, scene, dynamic=dynamic, dtype=dtype, record=True, **kw)
    for n in (chunks or [T]):
        ep.run(n)
    return ep.results()


def same(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True) if np.asarray(a).dtype.kind == "f" else \
        np.array_equal(a, b)


KEYS = ("q", "qdot", "traj", "steps_to_success", "min_clear_robots", "min_clear_scene", "nonfinite_steps")


def sensitivity(q0, goals, scene, dynamic, T, qd0):
    """How far the CPU loop moves from itself when its start state moves by one ulp."""
    ref = cpu_point_loop(q0, goals, scene, dynamic, T, qd0)["traj"]
    pert = cpu_point_loop(q0, goals, scene, dynamic, T, qd0, q_in=np.nextafter(q0, np.inf))["traj"]
    return np.abs(ref - pert).max()


@pytest.mark.parametrize("dynamic", [False, True])
def test_point_episodes_match_cpu_loop_f64(built, dynamic):
    """The example scene (jitter = 0) and 64 jittered scenes over 300 steps: q at every step to 1e-7, done_at and
    nonfinite_steps identical, clearances (functions of the state) to 1e-7.  A scene that drifts further must be
    sensitive: the CPU loop moves at least as far from itself under a 1-ulp change of its start state."""
    T = 300
    q0, goals, scene = m.scenarios.point_masses(65, seed=5, jitter=0.3)
    q0[0], goals[0] = m.scenarios.POINT_STARTS, m.scenarios.POINT_GOALS
    res = run(q0, goals, scene, dynamic, T)
    n_sens = 0
    for b in range(len(q0)):
        ref = cpu_point_loop(q0[b], goals[b], scene[b], dynamic, T)
        err = np.abs(res["traj"][b] - ref["traj"]).max()
        if err >= 1e-7:
            s = sensitivity(q0[b], goals[b], scene[b], dynamic, T, np.zeros((4, 3)))
            assert s >= err, (b, err, s)
            n_sens += 1
            continue
        assert res["steps_to_success"][b] == ref["done_at"], b
        assert res["nonfinite_steps"][b] == ref["nonfinite_steps"], b
        assert abs(res["min_clear_robots"][b] - ref["min_clear_robots"]) < 1e-7, b
        assert abs(res["min_clear_scene"][b] - ref["min_clear_scene"]) < 1e-7, b
    assert n_sens <= 3, n_sens
    print(f"dynamic={dynamic}: {len(q0) - n_sens}/{len(q0)} scenes within 1e-7 over {T} steps, {n_sens} shown sensitive; "
          f"success {res['success'].mean():.3f}")


def reach_scenes(B, R, seed):
    """B scenarios of R robots on a grid 1.5 apart (jittered by +-0.2) whose goals lie 0.5 from their starts, so most
    episodes succeed after 150-250 steps.  Scene (S = 3): a far sphere and two small trap spheres (radius 0.05) centred
    on the leaf point (x, y, 0.05) of a robot's start -- that robot's first action is 0/0, non-finite.  b % 3 == 1: robot 0
    is trapped; b % 3 == 2: robots 0 and R-1 are trapped in the same step (one counted step); otherwise the traps sit far
    away.  A trapped robot starts moving toward its goal at 0.3, so it coasts out of the trap and goes on."""
    rng = np.random.default_rng(seed)
    c = int(np.ceil(np.sqrt(R)))
    q0, goals, qd0 = np.zeros((B, R, 3)), np.zeros((B, R, 2)), np.zeros((B, R, 3))
    scene = np.zeros((B, 3, 4))
    scene[:, 0] = [40.0, 40.0, 0.0, 1.0]
    scene[:, 1] = [-40.0, 40.0, 0.05, 0.05]
    scene[:, 2] = [40.0, -40.0, 0.05, 0.05]
    for b in range(B):
        k = np.arange(R)
        q0[b, :, 0:2] = np.stack([1.5 * (k % c), 1.5 * (k // c)], axis=1) + rng.uniform(-0.2, 0.2, (R, 2))
        while True:
            ph = rng.uniform(0, 2 * np.pi, R)
            u = np.stack([np.cos(ph), np.sin(ph)], axis=1)
            g = q0[b, :, 0:2] + 0.5 * u
            d = np.linalg.norm(g[:, None] - g[None], axis=-1) + 10 * np.eye(R)
            if d.min() > 0.6:
                break
        goals[b] = g
        trapped = [] if b % 3 == 0 else ([0] if b % 3 == 1 else [0, R - 1])
        for n, i in enumerate(trapped):
            scene[b, 1 + n, 0:2] = q0[b, i, 0:2]
            qd0[b, i, 0:2] = 0.3 * u[i]
    return q0, goals, scene, qd0


@pytest.mark.parametrize("dynamic", [False, True])
@pytest.mark.parametrize("R", [2, 3, 4, 8])
def test_reaching_episodes_match_cpu_loop_f64(built, R, dynamic):
    """Episodes that succeed and episodes with non-finite steps, against the CPU loop: 12 scenarios (lane groups padded for
    R = 3, groups in the upper lanes of a warp), 250 steps run as run(100); run(150) -- a split before most done_at.  q to
    1e-7 at every step, done_at and nonfinite_steps identical, clearances to 1e-7; and the chunked run carries the
    bits of one run(250)."""
    B, T = 12, 250
    q0, goals, scene, qd0 = reach_scenes(B, R, seed=60 + R)
    res = run(q0, goals, scene, dynamic, T, qdot0=qd0, chunks=[100, 150])
    one = run(q0, goals, scene, dynamic, T, qdot0=qd0)
    for k in KEYS:
        assert same(res[k], one[k]), k
    for b in range(B):
        ref = cpu_point_loop(q0[b], goals[b], scene[b], dynamic, T, qd0[b])
        assert ref["nonfinite_steps"] == (0 if b % 3 == 0 else 1), b
        err = np.abs(res["traj"][b] - ref["traj"]).max()
        assert err < 1e-7, (b, err)
        assert res["steps_to_success"][b] == ref["done_at"], b
        assert res["nonfinite_steps"][b] == ref["nonfinite_steps"], b
        assert abs(res["min_clear_robots"][b] - ref["min_clear_robots"]) < 1e-7, b
        assert abs(res["min_clear_scene"][b] - ref["min_clear_scene"]) < 1e-7, b
    done = res["steps_to_success"]
    print(f"R={R} dynamic={dynamic}: done_at {sorted(done.tolist())}")
    assert (done > 100).sum() >= B // 3 and (done[1::3] >= 0).any()


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("dynamic", [False, True])
def test_one_step_equals_point_action_entry(built, dtype, dynamic):
    """From random states, n_steps = 1: (qdot1 - qdot0) / dt is mrf_point_action_dev's action for the same staged
    obstacles, within the rounding of the update; q1 = q0 + dt qdot1 as rounded in the entry's precision.  Both kernels
    inline the same point_action, but the compiler contracts a few products of the leaf algebra into FMAs differently at
    the two call sites: on a B200 about 98.5 % of the components of qdot1 equal qdot0 + dt a bit for bit, and the rest
    stay within 2.5 units of the update's rounding."""
    import torch
    B, R = 256, 4
    q0, goals, scene, qd0 = random_scenes(B, R, seed=21)
    qd0[:, :, 2] = np.random.default_rng(22).uniform(-0.5, 0.5, (B, R))
    q0[:, :, 2] = np.random.default_rng(23).uniform(-0.05, 0.05, (B, R))      # theta lands in the static spheres' z
    res = run(q0, goals, scene, dynamic, 1, dtype=dtype, qdot0=qd0)
    npt = np.float32 if dtype == "f32" else np.float64
    tdt = torch.float32 if dtype == "f32" else torch.float64
    dt = npt(default_config(1).dt)
    # the same obstacles staged for the one-robot entry: scene spheres, then the other robots ascending
    Ss, Sd = 6 + (0 if dynamic else R - 1), (R - 1 if dynamic else 0)
    rec, stat, dyn = np.zeros((B, R, 10)), np.zeros((B, R, Ss, 4)), np.zeros((B, R, max(Sd, 1), 7))
    for i in range(R):
        oth = [j for j in range(R) if j != i]
        rec[:, i, 0:3], rec[:, i, 3:6], rec[:, i, 6:8], rec[:, i, 8], rec[:, i, 9] = q0[:, i], qd0[:, i], goals[:, i], 1.0, 0.2
        stat[:, i, 0:6] = scene
        if dynamic:
            dyn[:, i, :, 0:2], dyn[:, i, :, 2:4], dyn[:, i, :, 6] = q0[:, oth, 0:2], qd0[:, oth, 0:2], 0.2
        else:
            stat[:, i, 6:, 0:3], stat[:, i, 6:, 3] = q0[:, oth], 0.2
    t = lambda a: torch.from_numpy(np.ascontiguousarray(np.moveaxis(a.reshape((B * R,) + a.shape[2:]), 0, -1))).to("cuda:0", dtype=tdt)
    fab = Fabrics(config=default_config(1))
    act = fab.point_action_dev(t(rec), t(stat), t(dyn) if dynamic else None)
    torch.cuda.synchronize()
    a = act.T.cpu().numpy().reshape(B, R, 3)
    fab.close()
    qd0_t, q0_t = qd0.astype(npt), q0.astype(npt)
    qd1, q1 = res["qdot"].astype(npt), res["q"].astype(npt)
    assert np.isfinite(a).all()
    ulp = np.finfo(npt).eps
    d = np.abs((qd1.astype(np.float64) - qd0_t) / dt - a)
    upd = 2 * ulp * (np.abs(qd0_t) + np.abs(qd1)) / dt + 2 * ulp * np.abs(a)      # rounding of the update
    exact = np.mean(qd1 == qd0_t + dt * a)
    print(f"{dtype} dynamic={dynamic}: qdot1 == qdot0 + dt a bit for bit on {exact:.4f} of components; "
          f"max |dqdot/dt - a| / update rounding {np.max(d / upd):.3g}; max rel {np.max(d / np.maximum(1, np.abs(a))):.3g}")
    assert (d <= 4 * upd).all() and exact >= 0.95
    assert np.max(d / np.maximum(1, np.abs(a))) <= (5e-6 if dtype == "f32" else 1e-14)    # measured 2.5e-6 / 6.1e-15
    assert np.array_equal(q1, q0_t + dt * qd1)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("dynamic", [False, True])
def test_chunking_is_invisible(built, dtype, dynamic):
    """run(7); run(13) gives the bits of run(20): state, metrics and trajectory."""
    q0, goals, scene = m.scenarios.point_masses(200, seed=31, jitter=0.4)
    a = run(q0, goals, scene, dynamic, 20, dtype=dtype)
    b = run(q0, goals, scene, dynamic, 20, dtype=dtype, chunks=[7, 13])
    for k in KEYS:
        assert same(a[k], b[k]), k
    assert b["steps"] == 20


@pytest.mark.parametrize("R", [2, 3, 4, 8])
def test_no_cross_talk(built, R):
    """Permuting the scenarios of a batch permutes the results bit for bit, and a batch whose size is not a multiple of the
    lane group (R padded to 2, 4, 8) or of the CTA agrees with scenarios run alone.  FP32 and FP64, both variants."""
    B = 37
    q0, goals, scene, qd0 = random_scenes(B, R, seed=40 + R)
    perm = np.random.default_rng(R).permutation(B)
    for dtype in ("f32", "f64"):
        for dynamic in (False, True):
            a = run(q0, goals, scene, dynamic, 40, dtype=dtype, qdot0=qd0)
            p = run(q0[perm], goals[perm], scene[perm], dynamic, 40, dtype=dtype, qdot0=qd0[perm])
            for k in KEYS:
                assert same(a[k][perm], p[k]), (dtype, dynamic, k)
            for b in (0, 17, B - 1):
                s = run(q0[b:b + 1], goals[b:b + 1], scene[b:b + 1], dynamic, 40, dtype=dtype, qdot0=qd0[b:b + 1])
                for k in KEYS:
                    assert same(a[k][b:b + 1], s[k]), (dtype, dynamic, b, k)


@pytest.mark.parametrize("dynamic", [False, True])
def test_fp32_coverage(built, dynamic):
    """FP32 against FP64 on 64 jittered example scenes after 300 steps: the share of scenarios whose positions agree to
    1e-3 and whose done_at agrees (a coverage statement, like DESIGN's FP32 accuracy paragraph)."""
    q0, goals, scene = m.scenarios.point_masses(64, seed=5, jitter=0.3)
    r64 = run(q0, goals, scene, dynamic, 300, dtype="f64")
    r32 = run(q0, goals, scene, dynamic, 300, dtype="f32")
    err = np.abs(r32["q"] - r64["q"]).max(axis=(1, 2))
    close, same_done = np.mean(err < 1e-3), np.mean(r32["steps_to_success"] == r64["steps_to_success"])
    print(f"dynamic={dynamic}: FP32 within 1e-3 of FP64 after 300 steps on {close:.3f} of scenes; done_at agrees on "
          f"{same_done:.3f}; median err {np.median(err):.2e}")
    assert close >= 0.9 and same_done >= 0.9
    q0, goals, scene = m.scenarios.point_masses_reach(64, seed=5)
    r64 = run(q0, goals, scene, dynamic, 300, dtype="f64")
    r32 = run(q0, goals, scene, dynamic, 300, dtype="f32")
    d64, d32 = r64["steps_to_success"], r32["steps_to_success"]
    same_done, n_done = np.mean(d32 == d64), int((d64 >= 0).sum())
    print(f"dynamic={dynamic}: reach workload, {n_done}/64 succeed in FP64 within 300 steps; FP32 done_at equal on "
          f"{same_done:.3f}, within 1 step on {np.mean(np.abs(d32 - d64) <= 1):.3f}")
    assert n_done >= 16 and same_done >= 0.9


def test_argument_checks(built):
    """Each MRF_EINVAL case of mrf_point_episode_run_dev_*, raised as MrfError."""
    q0, goals, scene = m.scenarios.point_masses(8, seed=1)
    ep = BatchedPointEpisodes(q0, goals, scene, dtype="f32")
    ep.run(1)
    base = ep._ep
    fn = lib().mrf_point_episode_run_dev_f32

    def call(n_steps=1, **fields):
        s = type(base).from_buffer_copy(base)
        for k, v in fields.items():
            setattr(s, k, v)
        rc = fn(ep.fab.handle.ptr, C.byref(s), ep.B, n_steps, None)
        assert rc == -1, (fields, n_steps, rc)                         # MRF_EINVAL
        with pytest.raises(MrfError):
            check(rc, "mrf_point_episode_run_dev")

    call(struct_size=base.struct_size - 8)
    call(n_robots=1)
    call(n_robots=9)
    call(n_scene=-1)
    call(n_scene=17)
    call(dynamic=2)
    for k in ("state", "goal", "weight", "radius", "scene", "time_step", "done_at", "nonfinite_steps", "min_clear_robots",
              "min_clear_scene"):
        call(**{k: None})
    call(n_steps=0)
    assert fn(ep.fab.handle.ptr, C.byref(base), 0, 1, None) == -1    # B = 0
    ok = type(base).from_buffer_copy(base)
    ok.scene, ok.n_scene = None, 0                                     # no scene: valid
    assert fn(ep.fab.handle.ptr, C.byref(ok), ep.B, 1, None) == 0
    q9 = np.zeros((2, 9, 3))
    q9[:, :, 0] = np.arange(9)
    with pytest.raises(MrfError):                                      # 9 robots: refused by the library
        BatchedPointEpisodes(q9, np.zeros((2, 9, 2)), None).run(1)
