"""FP32-only kernel paths held to a PER-SCENARIO bound at well-conditioned inputs.

The FP32 instantiations run code the FP64 kernels never run (paired point table, packed sphere_leaf2 / FFMA2 leaves,
the paired negated Cholesky, the Cody-Waite sincos, MUFU exp / tanh, the shared robot-robot leaves of the uniform
3-robot kernel, the obstacle-major accumulation and cp.async ring of action_kernel, kKeepJ8).  The long-horizon
statistical test (test_gpu_parity.py::test_rollout_f32_within_tolerance) covers stiff near-contact scenarios; here the
inputs are well conditioned BY CONSTRUCTION and the horizons short, so that every scenario can be held to a bound a few
times FP32 rounding:

- records from scenarios.generate(..., min_clearance=0.5), obstacles from helpers.random_obstacles (spheres with a
  normalised clearance below 0.5 pushed away) with non-zero velocity and acceleration;
- records and obstacles rounded to float32 first, so that both sides read identical values;
- a scenario is dropped only by a rule on float64 data (reference non-finite, or its robots' clearance along the
  reference trajectory below CLEAR_MARGIN); at least 95 % of the scenarios are kept;
- metric: per scenario, worst |got - ref| over its elements divided by max(1, max |ref|) (helpers.err_ps); EVERY kept
  scenario must be under the case's bound.
- reference: oracle O2; for the page-locked in-place path at B = 8193 the FP64 kernel on the same float32 inputs
  (pinned to O2 at 1e-9 by test_gpu_parity.py).

Bounds: 8x the worst per-scenario error measured on a B200 (1000 W) over seeds 0..4 of every case, see BOUND.
tools/fp32_mutants.py builds libraries with single arithmetic edits in FP32-only code and shows that these bounds fail
on each of them.
"""
import contextlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from multi_robot_fabrics_b200 import scenarios as sc
from multi_robot_fabrics_b200.api import Fabrics, to_soa
from multi_robot_fabrics_b200.spheres import sphere_offsets
from oracle import o2

from helpers import err_ps, oracle_actions, random_obstacles

DEV = "cuda:0"
SEEDS = (0, 1)
CLEAR_MARGIN = 0.25            # normalised clearance (scenarios.clearance) along the reference trajectory
MOUNT4 = [0.3, -0.6, 0.65]     # the fourth arm's base (the default one coincides with robot 0's)

# Worst per-scenario error measured on a B200 (1000 W power limit) over seeds 0..4 of every case of a family -> bound
# (8x, two significant digits).  Per-scenario metric of helpers.err_ps unless noted.
#   family (dispatch)                                                                     measured   bound
#   coupled, R <= 2: cooperative R2, throughput R1 / R2, link subsets R2, risk entry R2     9.2e-7   7.4e-6
#   coupled, R = 3, 4: cooperative R3 / R4 (+ estimate_goal 2, link subsets), throughput R4,
#     uniform 3-robot shared-leaf path (+ estimate_goal 1 / 2), risk entry R3                4.0e-6   3.2e-5
#   batch shapes B = 1, 31, 33 (throughput kernel and default dispatch)                    9.5e-7   7.6e-6
#   batch shapes B = 512 (cooperative / throughput), 513 (throughput)                      5.3e-6   4.3e-5
#   uniform tile with one fall-back scenario                                                7.4e-7   6.0e-6
#   the same scenario on the shared-leaf path and on the fall-back (one ulp of one radius)  5.5e-9   4.4e-8
#   static spheres, n_static 1 / 16                                                         1.4e-6   1.1e-5
#   page-locked in place, B = 8193, against the FP64 kernel                                 8.9e-6   7.1e-5
#   executed action, S <= 5 and the grasp planner                                           4.9e-7   3.9e-6
#   executed action, S = 12..192, robot_first, unequal radii, mode acc                      2.9e-6   2.4e-5
#   Cartesian rollouts, one robot per call and all robots in one launch                     7.7e-7   6.2e-6
#   kinematics x / v / a (absolute)                                                         9.0e-7   7.2e-6
#   obstacle staging (absolute)                                                             2.9e-7   2.4e-6
#   risk FP32 (relative to the scenario's largest risk), R = 2                              1.1e-6   9.0e-6
#   risk FP32, R = 3 (shared-leaf path and fall-back)                                       5.9e-6   4.7e-5
#   risk of the same scenario, shared-leaf path against fall-back                           9.6e-7   7.7e-6
BOUND = {
    "coupled-R12": 7.4e-6, "coupled-R34": 3.2e-5, "batch-small": 7.6e-6, "batch-large": 4.3e-5, "fallback": 6.0e-6,
    "fallback-same": 4.4e-8, "static": 1.1e-5, "inplace": 7.1e-5, "action-small": 3.9e-6, "action": 2.4e-5,
    "cart": 6.2e-6, "kin": 7.2e-6, "obst": 2.4e-6, "risk-R2": 9.0e-6, "risk-R3": 4.7e-5, "risk-same": 7.7e-6,
}
WORST = {}      # case id -> worst error seen in this process (read by the bound measurement)


def _check(case, e, bound_key):
    w = float(np.max(e))
    WORST[case] = max(WORST.get(case, 0.0), w)
    b = BOUND[bound_key]
    assert w < b, f"{case}: worst per-scenario error {w:.3e} exceeds the bound {b:.1e} ({w / b:.1f}x)"


@pytest.fixture(scope="module")
def fabs(built):
    d = {}
    yield d
    for f in d.values():
        f.close()


def get_fab(fabs, R, **kw):
    key = (R, tuple(sorted((k, repr(v)) for k, v in kw.items())))
    if key not in fabs:
        if R == 4 and "mount" not in kw:
            with mount4():
                kw["mount"] = [sc.mount_matrix(r) for r in range(4)]
        fabs[key] = Fabrics(R, device=0, **kw)
    return fabs[key]


@contextlib.contextmanager
def mount4():
    old = sc.MOUNT_XYZ[3].copy()
    sc.MOUNT_XYZ[3] = MOUNT4
    try:
        yield
    finally:
        sc.MOUNT_XYZ[3] = old


def ocfg_of(R, **kw):
    cfg = o2.default_config(R, **{k: v for k, v in kw.items() if k not in ("collision_links", "r_robots")})
    if "collision_links" in kw:
        o2.set_collision_links(cfg, kw["collision_links"])
    if R == 4:
        with mount4():
            for r in range(R):
                for i, v in enumerate(sc.mount_matrix(r).reshape(16)):
                    cfg.mount[r][i] = v
    return cfg


def f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def records(B, R, seed, **kw):
    if R == 4:
        with mount4():
            return f32(sc.generate(B, R, seed=seed, min_clearance=0.5, **kw))
    return f32(sc.generate(B, R, seed=seed, min_clearance=0.5, **kw))


def traj_clearance(rec, qN):
    """Worst normalised clearance (scenarios.clearance) over the initial state and every state of the trajectory."""
    R = rec.shape[1]
    ctx = mount4() if R == 4 else contextlib.nullcontext()
    with ctx:
        c = sc.clearance(rec)
        for k in range(qN.shape[2]):
            r = rec.copy()
            r[:, :, 0:7] = qN[:, :, k]
            with np.errstate(invalid="ignore"):
                c = np.minimum(c, np.nan_to_num(sc.clearance(r), nan=-np.inf))
    return c


def keep(ref_arrays, rec=None, qN=None):
    ok = np.ones(ref_arrays[0].shape[0], dtype=bool)
    for a in ref_arrays:
        ok &= np.isfinite(a).reshape(a.shape[0], -1).all(axis=1)
    if qN is not None:
        ok &= traj_clearance(rec, np.nan_to_num(qN)) >= CLEAR_MARGIN
    assert ok.mean() >= 0.95, f"only {ok.sum()} of {ok.size} scenarios kept"
    return ok


def dev(a, dt):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dtype=dt)


def host(t, *perm):
    return t.permute(*perm).double().cpu().numpy() if perm else t.double().cpu().numpy()


# ------------------------------------------------------------------------------------------- coupled rollouts
def roll_f32(fab, rec, N, coop=None):
    """mrf_rollout_dev_f32 with every output -> dict in record order (B, ...)."""
    import torch
    B, R = rec.shape[:2]
    t = lambda *s: torch.empty(s, dtype=torch.float32, device=DEV)
    qN, qdN, xee, ge = t(R, N, 7, B), t(R, N, 7, B), t(R, 3, B), t(3, B)
    if coop is not None:
        fab.handle.set_coop_max_batch(coop)
    try:
        avg = fab.rollout_dev(dev(to_soa(rec), torch.float32), N, x_ee=xee, goal_est=ge, qN=qN, qdN=qdN)
        torch.cuda.synchronize()
    finally:
        fab.handle.set_coop_max_batch(512)
    return dict(qN=host(qN, 3, 0, 1, 2), qdN=host(qdN, 3, 0, 1, 2), avg_vel=host(avg, 1, 0), x_ee=host(xee, 2, 0, 1),
                goal_est=host(ge, 1, 0))


def ref_rollout(ocfg, rec, N, est=0):
    return o2.rollout_rfcv(ocfg, rec, N, est_robot=1 if est else -1, use_jqd=est == 2, trajectories=True)


def coupled_err(got, ref, rec, est):
    keys = ["qN", "qdN", "avg_vel", "x_ee"] + (["goal_est"] if est else [])
    ok = keep([ref[k] for k in keys], rec, ref["qN"])
    return np.max([err_ps(got[k], ref[k]) for k in keys], axis=0), ok


# (id, R, kernel, B, estimate_goal, config overrides); kernel: "coop" = cooperative small-batch kernel, "thr" = throughput
# kernel (R = 3 with uniform radii: the uniform 3-robot kernel with the shared robot-robot leaves)
COUPLED = [
    ("coop-R2", 2, "coop", 64, 0, {}),
    ("coop-R3", 3, "coop", 64, 0, {}),
    ("coop-R4", 4, "coop", 64, 0, {}),
    ("thr-R1", 1, "thr", 64, 0, {}),
    ("thr-R2", 2, "thr", 64, 0, {}),
    ("thr-R4", 4, "thr", 64, 0, {}),
    ("pair-R3", 3, "thr", 96, 0, {}),
    ("pair-R3-est1", 3, "thr", 96, 1, {}),
    ("pair-R3-est2", 3, "thr", 96, 2, {}),
    ("coop-R3-est2", 3, "coop", 64, 2, {}),
    ("links-R2", 2, "thr", 64, 0, {"collision_links": [[3, 6, 8], [1, 2, 4, 7]]}),
    ("links-R3-coop", 3, "coop", 64, 0, {"collision_links": [[5], [3, 4, 5, 6, 7], [1, 2, 3, 4, 5, 6, 7, 8]]}),
]


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("case,R,kernel,B,est,kw", COUPLED, ids=[c[0] for c in COUPLED])
def test_coupled_rollout_f32(fabs, case, R, kernel, B, est, kw, N, seed):
    """mrf_rollout_dev_f32: qN, qdN, avg_vel, x_ee (and goal_est with estimate_goal) against O2 per scenario."""
    rec = records(B, R, 10 * seed + R)
    fab = get_fab(fabs, R, estimate_goal=est, **kw)
    got = roll_f32(fab, rec, N, coop=0 if kernel == "thr" else 1 << 20)
    e, ok = coupled_err(got, ref_rollout(ocfg_of(R, **kw), rec, N, est), rec, est)
    _check(f"coupled/{case}/N{N}", e[ok], "coupled-R12" if R <= 2 else "coupled-R34")


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("B", [1, 31, 33, 512, 513])
def test_coupled_rollout_f32_batch_shapes(fabs, B, seed):
    """Partial tiles of the throughput kernel, and both sides of the cooperative threshold (B <= 512: cooperative
    kernel, 513: throughput kernel) with the default dispatch; 3 robots, estimate_goal = 1, N = 3."""
    R, N = 3, 3
    rec = records(B, R, 20 + seed)
    fab = get_fab(fabs, R, estimate_goal=1)
    ref = ref_rollout(ocfg_of(R), rec, N, 1)
    for coop in (0, None):
        e, ok = coupled_err(roll_f32(fab, rec, N, coop=coop), ref, rec, 1)
        _check(f"batch/B{B}/{'thr' if coop == 0 else 'default'}", e[ok], "batch-small" if B < 512 else "batch-large")


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("N", [1, 3])
def test_pair_path_fallback_scenario(fabs, N, seed):
    """Uniform 3-robot kernel: one scenario with unequal body radii (link3 one float ulp larger) inside a tile of uniform
    ones takes the per-scenario fall-back (every leaf evaluated by its own robot); its neighbours stay on the shared-leaf
    path -- their results are bitwise those of the same batch without the odd scenario -- and every scenario is within
    the bound of O2."""
    R, B, odd = 3, 64, 37
    rec = records(B, R, 30 + seed)
    odd_rec = rec.copy()
    odd_rec[odd, 1, o2.RB] = float(np.nextafter(np.float32(rec[odd, 1, o2.RB]), np.float32(1)))
    fab = get_fab(fabs, R)
    base = roll_f32(fab, rec, N, coop=0)
    got = roll_f32(fab, odd_rec, N, coop=0)
    nb = np.arange(B) != odd
    for k in base:
        assert np.array_equal(got[k][nb], base[k][nb], equal_nan=True), k
    e, ok = coupled_err(got, ref_rollout(ocfg_of(R), odd_rec, N), odd_rec, 0)
    assert ok[odd]
    _check(f"fallback/N{N}", e[ok], "fallback")
    # the same scenario on the two paths (its records differ by one ulp of one radius)
    _check(f"fallback/pair-vs-fallback/N{N}", err_ps(got["qdN"][odd:odd + 1], base["qdN"][odd:odd + 1]), "fallback-same")


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("R,S", [(2, 1), (2, 16), (3, 1), (3, 16)])
def test_static_sphere_rollout_f32(fabs, R, S, N, seed):
    """mrf_rollout_static_dev_f32 (generic throughput kernel with static spheres at rest) against O2 per scenario."""
    import torch
    B = 48
    rng = np.random.default_rng(40 + seed)
    rec = records(B, R, 40 + seed)
    stat = np.zeros((B, R, S, 4))
    stat[..., 0:3] = rng.uniform([-0.6, -1.2, 0.9], [1.6, 1.2, 2.0], size=(B, R, S, 3))
    stat[..., 3] = rng.uniform(0.05, 0.12, size=(B, R, S))
    for r in range(R):                                   # spheres near a link of their robot: pushed out of the way
        pos = sc.link_positions(rec[:, r, 0:7], sc.mount_matrix(r))
        d = np.linalg.norm(stat[:, r, :, None, 0:3] - pos[:, None], axis=-1).min(axis=-1)
        stat[:, r, :, 2] += np.where(d / (stat[:, r, :, 3] + 0.08) - 1.0 < 0.5, 1.5, 0.0)
    stat = f32(stat)
    ocfg = o2.default_config(R)
    ref = {k: np.zeros(s) for k, s in (("qN", (B, R, N, 7)), ("qdN", (B, R, N, 7)), ("avg_vel", (B, R)), ("x_ee", (B, R, 3)))}
    for b in range(B):
        ref["qN"][b], ref["qdN"][b], ref["avg_vel"][b], ref["x_ee"][b] = o2.rollout_jointspace_static(
            ocfg, rec[b], N, stat[b, :, :, 0:3], stat[b, :, :, 3])
    fab = get_fab(fabs, R)
    t = lambda *s: torch.empty(s, dtype=torch.float32, device=DEV)
    qN, qdN, xee = t(R, N, 7, B), t(R, N, 7, B), t(R, 3, B)
    avg = fab.rollout_static_dev(dev(to_soa(rec), torch.float32), dev(stat.transpose(2, 3, 1, 0), torch.float32), N,
                                 x_ee=xee, qN=qN, qdN=qdN)
    torch.cuda.synchronize()
    got = dict(qN=host(qN, 3, 0, 1, 2), qdN=host(qdN, 3, 0, 1, 2), avg_vel=host(avg, 1, 0), x_ee=host(xee, 2, 0, 1))
    ok = keep(list(ref.values()), rec, ref["qN"])
    e = np.max([err_ps(got[k], ref[k]) for k in ref], axis=0)
    _check(f"static/R{R}/S{S}/N{N}", e[ok], "static")


def test_page_locked_in_place_rollout_f32(fabs):
    """B = 8193 page-locked float32 records read in place (rollout_kernel<float,3,uniform,AOS>) against the FP64 kernel
    on the same float32 inputs: avg_vel, x_ee, goal_est per scenario."""
    import torch
    R, N, B = 3, 3, 8193
    rec = records(B, R, 50)
    fab = get_fab(fabs, R, estimate_goal=1)
    ref = fab.rollout_host(rec, N, dtype="f64", trajectories=True)
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    out = {"avg_vel": pin(np.zeros((B, R), np.float32)), "x_ee": pin(np.zeros((B, R, 3), np.float32)),
           "goal_est": pin(np.zeros((B, 3), np.float32))}
    n0 = fab.handle.launches
    fab.rollout_host(pin(rec.astype(np.float32)), N, dtype="f32", out=out)
    assert fab.handle.launches - n0 == 1                                 # the in-place kernel, no staging
    keys = ("avg_vel", "x_ee", "goal_est")
    ok = keep([ref[k] for k in keys + ("qN",)], rec, ref["qN"])
    e = np.max([err_ps(out[k], ref[k]) for k in keys], axis=0)
    _check("inplace/B8193", e[ok], "inplace")


# ------------------------------------------------------------------------------------------- executed action
# (id, R, n_rob, robot_first, S, variant)
ACTION = [(f"S{S}", 2, 2, 0, S, None) for S in (1, 2, 3, 5, 31, 64)] + [
    ("R4-S192", 4, 4, 0, 192, None),          # 8 spheres per link of the three other robots
    ("robot_first1", 3, 2, 1, 12, None),
    ("body_radii", 2, 2, 0, 12, "body_radii"),
    ("obst_radii", 2, 2, 0, 13, "obst_radii"),
    ("grasp", 2, 2, 0, 12, "grasp"),
    ("acc", 2, 2, 0, 12, "acc"),
]


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("case,R,n_rob,robot_first,S,variant", ACTION, ids=[a[0] for a in ACTION])
def test_action_f32(fabs, case, R, n_rob, robot_first, S, variant, seed):
    """mrf_action_dev_f32 (obstacle-major packed accumulation, cp.async ring of S spheres, kKeepJ8) against O2 per
    scenario; B = 50 (B * n_rob not a multiple of the 128-thread block)."""
    import torch
    B = 50
    rng = np.random.default_rng(60 + seed)
    if R == 4:   # the executed action of each robot is independent of the others: two 2-robot batches side by side
        rec = np.concatenate([records(B, 2, 60 + seed, weight_goal_1=20.0), records(B, 2, 70 + seed, weight_goal_1=20.0)], 1)
    else:
        rec = records(B, R, 60 + seed, weight_goal_1=20.0)[:, robot_first:robot_first + n_rob]
    if variant == "body_radii":
        rec[:, :, o2.RB:o2.RB + 6] = f32([0.08, 0.07, 0.09, 0.06, 0.08, 0.1])
    with mount4() if R == 4 else contextlib.nullcontext():
        obst = random_obstacles(rng, B, n_rob, S, rec, robot_first=robot_first)
    if variant == "obst_radii":
        obst[..., 9] = rng.uniform(0.05, 0.12, size=obst.shape[:3])
    obst = f32(obst)
    kw = {"grasp": dict(has_collision_links=0), "acc": dict(mode=0)}.get(variant, {})
    fab = get_fab(fabs, R, **kw)
    act = fab.action_dev(dev(to_soa(rec), torch.float32), dev(obst.transpose(2, 3, 1, 0), torch.float32),
                         robot_first=robot_first)
    torch.cuda.synchronize()
    got = host(act, 2, 1, 0)
    ref = oracle_actions(rec, obst, robot_first=robot_first, **kw) if R < 4 else _actions4(rec, obst)
    ok = keep([ref])
    _check(f"action/{case}", err_ps(got, ref)[ok], "action-small" if S <= 5 or variant == "grasp" else "action")


def _actions4(rec, obst):
    cfg = ocfg_of(4)
    out = np.full(rec.shape[:2] + (7,), np.nan)
    for b in range(rec.shape[0]):
        for r in range(4):
            o = obst[b, r]
            try:
                out[b, r] = o2.action(cfg, r, rec[b, r], o[:, 0:3], o[:, 3:6], o[:, 6:9], o[:, 9])
            except FloatingPointError:
                pass
    return out


# ------------------------------------------------------------------------------------------- Cartesian rollouts
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("S", [1, 5, 16])
def test_cartesian_rollout_f32(fabs, S, N, seed):
    """mrf_rollout_cart_dev_f32 (one robot per call) and mrf_rollout_cart_all_dev_f32 (every robot in one launch) against
    o2.rollout_cartesian per robot and scenario: the obstacles move with constant velocity, x + k dt v at step k."""
    import torch
    R, B = 2, 48
    rng = np.random.default_rng(80 + seed)
    rec = records(B, R, 80 + seed, weight_goal_1=20.0)
    obst = f32(random_obstacles(rng, B, R, S, rec))
    ocfg = o2.default_config(R)
    ref = {k: np.zeros(s) for k, s in (("qN", (B, R, N, 7)), ("qdN", (B, R, N, 7)), ("avg_vel", (B, R)))}
    for b in range(B):
        for r in range(R):
            o = obst[b, r]
            ref["qN"][b, r], ref["qdN"][b, r], ref["avg_vel"][b, r] = o2.rollout_cartesian(
                ocfg, r, rec[b, r], o[:, 0:3], o[:, 3:6], o[:, 9], N)
    fab = get_fab(fabs, R)
    t = lambda *s: torch.empty(s, dtype=torch.float32, device=DEV)
    d_rec, d_obst = dev(to_soa(rec), torch.float32), dev(obst.transpose(2, 3, 1, 0), torch.float32)
    one = {k: np.zeros_like(v) for k, v in ref.items()}
    for r in range(R):
        qN, qdN = t(N, 7, B), t(N, 7, B)
        avg = fab.rollout_cart_dev(r, d_rec[:, r].contiguous(), d_obst[:, :, r].contiguous(), N, qN=qN, qdN=qdN)
        torch.cuda.synchronize()
        one["qN"][:, r], one["qdN"][:, r], one["avg_vel"][:, r] = host(qN, 2, 0, 1), host(qdN, 2, 0, 1), host(avg)
    qN, qdN = t(R, N, 7, B), t(R, N, 7, B)
    avg = fab.rollout_cart_all_dev(d_rec, d_obst, N, qN=qN, qdN=qdN)
    torch.cuda.synchronize()
    allr = dict(qN=host(qN, 3, 0, 1, 2), qdN=host(qdN, 3, 0, 1, 2), avg_vel=host(avg, 1, 0))
    ok = keep(list(ref.values()))
    for name, got in (("one", one), ("all", allr)):
        e = np.max([err_ps(got[k], ref[k]) for k in ref], axis=0)
        _check(f"cart/{name}/S{S}/N{N}", e[ok], "cart")


# ------------------------------------------------------------------------------------------- kinematics, obstacle staging
@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("R", [1, 2, 3, 4])
def test_kinematics_f32(fabs, R, seed):
    """mrf_kinematics_dev_f32: x, v and a = jdot_ref_sign * Jdot qdot of the 8 links against O2 (absolute: metres)."""
    import torch
    B = 64
    rec = records(B, R, 90 + seed)
    fab = get_fab(fabs, R)
    x, v, a = fab.kinematics_dev(dev(rec[:, :, 0:7].transpose(2, 1, 0), torch.float32),
                                 dev(rec[:, :, 7:14].transpose(2, 1, 0), torch.float32))
    torch.cuda.synchronize()
    got = np.stack([host(x, 3, 2, 0, 1), host(v, 3, 2, 0, 1), host(a, 3, 2, 0, 1)], axis=2)      # B,R,3,8,3
    ocfg = ocfg_of(R)
    ref = np.zeros_like(got)
    for b in range(B):
        for r in range(R):
            xx, vv, cc, _ = o2.kinematics(ocfg, r, rec[b, r, 0:7], rec[b, r, 7:14])
            ref[b, r] = xx, vv, -cc
    e = np.abs(got - ref).reshape(B, -1).max(axis=1)
    _check(f"kin/R{R}", e, "kin")


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("vel_mode", [0, 1])
@pytest.mark.parametrize("n", [1, 4, 8])
@pytest.mark.parametrize("R", [2, 3, 4])
def test_obstacles_f32(fabs, R, n, vel_mode, seed):
    """mrf_obstacles_dev_f32: the other robots' collision spheres of every ego robot (8 n (R-1) records) and the sphere
    positions / velocities against o2.obstacle_lists and o2.spheres (absolute)."""
    import torch
    B = 32
    rec = records(B, R, 100 + seed)
    fab = get_fab(fabs, R)
    t = lambda *s: torch.empty(s, dtype=torch.float32, device=DEV)
    sx, sv = t(8 * n, 3, R, B), t(8 * n, 3, R, B)
    obst = fab.obstacles_dev(dev(rec[:, :, 0:7].transpose(2, 1, 0), torch.float32),
                             dev(rec[:, :, 7:14].transpose(2, 1, 0), torch.float32), n_per_link=n, vel_mode=vel_mode,
                             spheres_x=sx, spheres_v=sv)
    torch.cuda.synchronize()
    got, gx, gv = host(obst, 3, 2, 0, 1), host(sx, 3, 2, 0, 1), host(sv, 3, 2, 0, 1)
    ocfg, off = ocfg_of(R), sphere_offsets(n)
    e = np.zeros(B)
    for b in range(B):
        lists = o2.obstacle_lists(ocfg, rec[b, :, 0:7], rec[b, :, 7:14], off, vel_mode=vel_mode)
        for r in range(R):
            x, vo, vs = o2.spheres(ocfg, r, rec[b, r, 0:7], rec[b, r, 7:14], off)
            e[b] = max(e[b], np.abs(got[b, r] - lists[r]).max(), np.abs(gx[b, r] - x).max(),
                       np.abs(gv[b, r] - (vs if vel_mode else vo)).max())
    _check(f"obst/R{R}/n{n}/v{vel_mode}", e, "obst")


# ------------------------------------------------------------------------------------------- risk
def risk_ref(ocfg, rec, qN, qdN):
    """Float64 restatement of the stiffness indicator `risk` of mrf_rollout_risk_dev_* on a reference trajectory.

    Per robot, the maximum over the horizon steps k = 0..N-1 of the summed collision-leaf metric sum trace(A_e): the
    state of step k is the one the step's action is evaluated at, q = qN[k] (after the position update) with the velocity
    of the previous step's action (the record's qdot at k = 0); the end-effector FK at the measured state (before step
    0) is not a step.  Per ego collision link l in 3..8 (bit l-1 of the robot's collision-link mask; none at all with
    has_collision_links = 0) with body radius rb_l:
      - a sphere leaf 0.02 / (x^4 rho^2) for every collision link l' of every other robot (bit l'-1 of that robot's mask),
        x = |p_l - p_l'| / rho - 1, rho = r_robots[j][l'] + rb_l;
      - the plane leaf 0.2 s / x^2, x = n.p_l + d - rb_l with the unit normal of constraint_0, gate s = 1 when
        n.v_l < 0, 0 when > 0, 1/2 when = 0.
    link1 / link2 and link5 / link6 share a point: the kernel's weight-2 merged entry (equal radii) is the sum of the two
    entries here; with unequal radii it evaluates both, as here.  Joint-limit and attractor leaves do not count."""
    B, R, N = qN.shape[:3]
    mask = [int(ocfg.link_mask[r]) if ocfg.has_collision_links else 0 for r in range(R)]
    out = np.zeros((B, R))
    for b in range(B):
        for k in range(N):
            kin = [o2.kinematics(ocfg, r, qN[b, r, k], rec[b, r, 7:14] if k == 0 else qdN[b, r, k - 1])[:2] for r in range(R)]
            for r in range(R):
                con = rec[b, r, o2.CON:o2.CON + 4]
                nh, dn = con[0:3] / np.linalg.norm(con[0:3]), con[3] / np.linalg.norm(con[0:3])
                tot = 0.0
                for l in range(3, 9):
                    if not (mask[r] >> (l - 1)) & 1:
                        continue
                    p, v, rb = kin[r][0][l - 1], kin[r][1][l - 1], rec[b, r, o2.RB + l - 3]
                    for j in range(R):
                        if j == r:
                            continue
                        for lo in range(1, 9):
                            if (mask[j] >> (lo - 1)) & 1:
                                rho = ocfg.r_robots[j][lo - 1] + rb
                                x = np.linalg.norm(p - kin[j][0][lo - 1]) / rho - 1.0
                                tot += 0.02 / (x ** 4 * rho ** 2)
                    xp, xd = nh @ p + dn - rb, nh @ v
                    s = 1.0 if xd < 0 else (0.0 if xd > 0 else 0.5)
                    tot += 0.2 * s / xp ** 2
                out[b, r] = max(out[b, r], tot)
    return out


def roll_risk(fab, rec, N, dt):
    import torch
    B, R = rec.shape[:2]
    t = lambda *s: torch.empty(s, dtype=dt, device=DEV)
    xee, risk = t(R, 3, B), t(R, B)
    avg = fab.rollout_dev(dev(to_soa(rec), dt), N, x_ee=xee, risk=risk)
    torch.cuda.synchronize()
    return host(risk, 1, 0), host(avg, 1, 0), host(xee, 2, 0, 1)


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("N", [1, 3])
@pytest.mark.parametrize("R", [2, 3])
def test_risk_against_restatement(fabs, R, N, seed):
    """risk of mrf_rollout_risk_dev_*: FP64 against risk_ref on the oracle trajectory to 1e-9 relative per scenario;
    FP32 within its bound (R = 3: the shared-leaf path of the uniform 3-robot kernel; R = 2 and a second tile of the
    same scenarios with one body radius one ulp larger: every leaf evaluated by its own robot), and the same scenario on
    the two paths against each other.  avg_vel and x_ee of the risk entry against O2 as the coupled rollouts."""
    import torch
    B = 32
    rec = records(B, R, 110 + seed)
    if R == 3:     # tile 2: the same scenarios on the per-scenario fall-back
        alt = rec.copy()
        alt[:, 2, o2.RB + 5] = f32(np.nextafter(np.float32(rec[:, 2, o2.RB + 5]), np.float32(1)))
        rec = np.concatenate([rec, alt])
    ocfg = ocfg_of(R)
    ref = ref_rollout(ocfg, rec, N)
    ok = keep([ref["qN"], ref["qdN"], ref["avg_vel"]], rec, ref["qN"])
    rref = risk_ref(ocfg, rec, ref["qN"], ref["qdN"])
    fab = get_fab(fabs, R)
    r64, _, _ = roll_risk(fab, rec, N, torch.float64)
    rel = np.abs(r64 - rref).max(axis=1) / np.abs(rref).max(axis=1)
    assert (rref > 0).all() and rel[ok].max() < 1e-9, rel[ok].max()
    r32, avg, xee = roll_risk(fab, rec, N, torch.float32)
    e = np.abs(r32 - rref).max(axis=1) / np.abs(rref).max(axis=1)
    _check(f"risk/f32/R{R}/N{N}", e[ok], f"risk-R{R}")
    _check(f"coupled/risk-entry/R{R}/N{N}", np.maximum(err_ps(avg, ref["avg_vel"]), err_ps(xee, ref["x_ee"]))[ok], "coupled-R12" if R <= 2 else "coupled-R34")
    if R == 3:
        both = ok[:B] & ok[B:]
        e = np.abs(r32[:B] - r32[B:]).max(axis=1) / np.abs(rref[:B]).max(axis=1)
        _check(f"risk/pair-vs-fallback/N{N}", e[both], "risk-same")
