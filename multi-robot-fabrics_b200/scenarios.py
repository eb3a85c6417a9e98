"""Synthetic multi-Panda scenarios (SURVEY.md section 8d) -- host-side input generation for tests and bench.py.

Distributions: q uniform inside the joint limits shrunk by 0.15 rad, qdot uniform in +-0.5 x the velocity limits
(examples/example_pandas_Jointspace.py:221), goals uniform in the box spanned by the reference's start goals
(examples/parameters_manipulators.py:126-132), weight_goal_0 in {2,3} (state_machine / deadlock_prevention.py:23-24),
weight_goal_1 = 10 for rollouts (example_pandas_Jointspace.py:43) or 20 for the executed action (:427), radii 0.08,
plane constraint (0,0,1,-0.65).  Scenarios whose initial configuration has a normalised sphere clearance below
`min_clearance` (default 0.25: the leaf metric 0.02/x^4 and force ~1/x^8 make closer starts numerically stiff
under the reference's explicit dt = 0.01 integration), or a sphere closer than that to the table plane, are redrawn (keeps the leaf metrics bounded).
"""
from __future__ import annotations

import math

import numpy as np

from ._lib import ANG, CON, G0, G1, G2, Q, QD, RB, REC, W0, W1, W2

PANDA_LIMITS = np.array([[-2.8973, 2.8973], [-1.7628, 1.7628], [-2.8973, 2.8973], [-3.0718, -0.0698],
                         [-2.8973, 2.8973], [-0.0175, 3.7525], [-2.8973, 2.8973]])
VEL_LIMITS = np.array([2.175, 2.175, 2.175, 2.175, 2.61, 2.61, 2.61])
ROT_PANDA = np.array([[0.0, 0.0, -1.0], [0.0, 1.0, 0.0], [1.0, 0.0, 0.0]])   # parameters_manipulators.py:121
MOUNT_XYZ = np.array([[0.0, 0.0, 0.65], [1.0, 0.0, 0.65], [0.7, 0.6, 0.65], [0.0, 0.0, 0.65]])
MOUNT_YAW = np.array([0.0, math.pi, math.pi, 0.0])      # example_pandas_Jointspace.py:108-110: pi for robots 1, 2
POS0_2 = np.array([1.125, 0.19, 0.12, -1.66, -0.0, 1.88, np.pi / 4])          # parameters_manipulators.py:93

_JXYZ = np.array([[0, 0, 0.333], [0, 0, 0], [0, -0.316, 0], [0.0825, 0, 0], [-0.0825, 0.384, 0], [0, 0, 0],
                  [0.088, 0, 0]], dtype=np.float64)
_JROLL = np.array([0.0, -1.0, 1.0, 1.0, -1.0, 1.0, 1.0]) * (math.pi / 2)


def mount_matrix(robot: int) -> np.ndarray:
    T = np.eye(4)
    c, s = math.cos(MOUNT_YAW[robot]), math.sin(MOUNT_YAW[robot])
    T[0:2, 0:2] = [[c, -s], [s, c]]
    T[0:3, 3] = MOUNT_XYZ[robot]
    return T


def link_positions(q: np.ndarray, mount: np.ndarray) -> np.ndarray:
    """World origins of panda_link1..8 for q of shape (..., 7) -> (..., 8, 3) (numpy, for rejection only)."""
    q = np.asarray(q, dtype=np.float64)
    shp = q.shape[:-1]
    R = np.broadcast_to(mount[:3, :3], shp + (3, 3)).copy()
    p = np.broadcast_to(mount[:3, 3], shp + (3,)).copy()
    out = np.zeros(shp + (8, 3))
    for i in range(7):
        p = p + R @ _JXYZ[i]
        cr, sr = math.cos(_JROLL[i]), math.sin(_JROLL[i])
        Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
        cq, sq = np.cos(q[..., i]), np.sin(q[..., i])
        Rz = np.zeros(shp + (3, 3))
        Rz[..., 0, 0], Rz[..., 0, 1], Rz[..., 1, 0], Rz[..., 1, 1], Rz[..., 2, 2] = cq, -sq, sq, cq, 1.0
        R = R @ Rx @ Rz
        out[..., i, :] = p
    out[..., 7, :] = p + R @ np.array([0.0, 0.0, 0.107])
    return out


def _draw(rng, n, n_robots, weight_goal_1):
    rec = np.zeros((n, n_robots, REC))
    lo, hi = PANDA_LIMITS[:, 0] + 0.15, PANDA_LIMITS[:, 1] - 0.15
    rec[..., Q:Q + 7] = rng.uniform(lo, hi, size=(n, n_robots, 7))
    rec[..., QD:QD + 7] = rng.uniform(-0.5, 0.5, size=(n, n_robots, 7)) * VEL_LIMITS
    rec[..., G0:G0 + 3] = rng.uniform([0.2, -0.6, 0.8], [0.8, 0.6, 1.25], size=(n, n_robots, 3))
    rec[..., W0] = rng.choice([2.0, 3.0], size=(n, n_robots))
    rec[..., G1:G1 + 3] = [0.107, 0.0, 0.0]
    rec[..., W1] = weight_goal_1
    rec[..., G2] = math.pi / 4
    rec[..., W2] = 1.0
    rec[..., ANG:ANG + 9] = ROT_PANDA.reshape(9)
    rec[..., CON:CON + 4] = [0.0, 0.0, 1.0, -0.65]
    rec[..., RB:RB + 6] = 0.08
    return rec


def clearance(rec: np.ndarray, radius: float = 0.08, z_table: float = 0.65) -> np.ndarray:
    """min over sphere pairs of |d|/(2 r) - 1 and over spheres of (z - z_table - r); per scenario."""
    n, R, _ = rec.shape
    pos = np.stack([link_positions(rec[:, r, Q:Q + 7], mount_matrix(r)) for r in range(R)], axis=1)  # n,R,8,3
    c = np.full(n, np.inf)
    for a in range(R):
        for b in range(a + 1, R):
            d = np.linalg.norm(pos[:, a, :, None, :] - pos[:, b, None, :, :], axis=-1)
            c = np.minimum(c, d.reshape(n, -1).min(axis=1) / (2 * radius) - 1.0)
    zc = (pos[:, :, 2:, 2] - z_table - radius).reshape(n, -1).min(axis=1)   # links 3..8 own plane leaves
    return np.minimum(c, zc)


def generate(n: int, n_robots: int, seed: int = 0, min_clearance: float = 0.25, weight_goal_1: float = 10.0) -> np.ndarray:
    """(n, n_robots, 44) float64 records, PCG64(seed)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = np.zeros((n, n_robots, REC))
    have = 0
    drawn = 0
    while have < n:
        m = max(256, int((n - have) * 2.0))
        rec = _draw(rng, m, n_robots, weight_goal_1)
        drawn += m
        if drawn > 200 * n + 100000 and have < 0.01 * drawn:
            raise ValueError(f"min_clearance={min_clearance} rejects (almost) every scenario (accepted {have} of {drawn})")
        ok = clearance(rec) >= min_clearance
        rec = rec[ok][: n - have]
        out[have:have + len(rec)] = rec
        have += len(rec)
    return out


def obstacles_from_positions(x, v=None, a=None, radius=0.08) -> np.ndarray:
    """Pack (.., S, 3) positions [velocities, accelerations] into (.., S, 10) obstacle records."""
    x = np.asarray(x, dtype=np.float64)
    o = np.zeros(x.shape[:-1] + (10,))
    o[..., 0:3] = x
    if v is not None:
        o[..., 3:6] = v
    if a is not None:
        o[..., 6:9] = a
    o[..., 9] = radius
    return o


def pick_and_place_layout(rec: np.ndarray, n_blocks: int = 2, seed: int = 0, spread: float = 0.12, drop: float = 0.16):
    """A synthetic pick-and-place task for episodes.BatchedEpisodes(blocks=, start_goal=): every robot's start goal is
    its hand position in `rec` (B,R,44) and its blocks rest `drop` below that height, uniformly within +-`spread` in x, y
    (the reference spreads cubes over the table around the start goals, create_simulation_manipulators.py:39-63).
    -> blocks (B, n_blocks, R, 3), start_goal (B, R, 3)."""
    B, R = rec.shape[:2]
    rng = np.random.Generator(np.random.PCG64(seed))
    start = np.zeros((B, R, 3))
    for r in range(R):
        start[:, r] = link_positions(rec[:, r, Q:Q + 7], mount_matrix(r))[:, 7]
    blocks = start[:, None, :, :] + np.stack([rng.uniform(-spread, spread, (B, n_blocks, R)),
                                              rng.uniform(-spread, spread, (B, n_blocks, R)),
                                              np.full((B, n_blocks, R), -drop)], axis=-1)
    return blocks, start


# ---- point masses (examples/example_pointmasses_static.py, _dynamic.py): 4 point robots swap sides between 6 spheres
POINT_SCENE = np.array([[1, 1.25, 0], [1, 3.75, 0], [1, -1.25, 0], [-1.1, 0, 0], [-1.1, 2.5, 0], [-1.1, -2.5, 0]], float)
POINT_SCENE_RADIUS = 1.0
POINT_STARTS = np.array([[-2.5, 0.01, 0.0], [-2.5, -2.49, 0.0], [2.5, 1.26, 0.0], [2.5, 3.74, 0.0]])
POINT_GOALS = np.array([[1.5, 3.76], [1.5, 1.26], [-2.5, 0.01], [-2.5, -2.49]])
POINT_RADIUS = 0.2


def point_masses(B: int, seed: int = 0, jitter: float = 0.0):
    """The point-mass examples' scene for episodes.BatchedPointEpisodes: 6 scene spheres of radius 1.0, 4 robots of radius
    0.2 and their start / goal swap pairs.  With jitter > 0 every scenario's starts and goals move by uniform offsets in
    [-jitter, jitter] in x and y (PCG64(seed)); a draw whose start has a robot in contact with another robot (x-y) or with
    a scene sphere (the collision leaf's distance from (x, y, 0.05)) is redrawn.  jitter = 0 is the example itself.
    -> q0 (B,4,3), goals (B,4,2), scene (B,6,4)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    q0 = np.broadcast_to(POINT_STARTS, (B, 4, 3)).copy()
    goals = np.broadcast_to(POINT_GOALS, (B, 4, 2)).copy()
    if jitter > 0:
        todo = np.arange(B)
        while len(todo):
            n = len(todo)
            q = np.broadcast_to(POINT_STARTS, (n, 4, 3)).copy()
            q[:, :, 0:2] += rng.uniform(-jitter, jitter, (n, 4, 2))
            g = POINT_GOALS + rng.uniform(-jitter, jitter, (n, 4, 2))
            ok = point_start_clearance(q) > 0
            q0[todo[ok]], goals[todo[ok]] = q[ok], g[ok]
            todo = todo[~ok]
    scene = np.zeros((B, len(POINT_SCENE), 4))
    scene[:, :, 0:3] = POINT_SCENE
    scene[:, :, 3] = POINT_SCENE_RADIUS
    return q0, goals, scene


def point_start_clearance(q0: np.ndarray, radius: float = POINT_RADIUS) -> np.ndarray:
    """min over robot pairs of the x-y clearance and over robots and scene spheres of the leaf clearance, per scenario."""
    p = q0[:, :, 0:2]
    d = np.linalg.norm(p[:, :, None, :] - p[:, None, :, :], axis=-1) - 2 * radius
    n = q0.shape[1]
    d[:, np.arange(n), np.arange(n)] = np.inf
    x = np.concatenate([p, np.full(p.shape[:2] + (1,), 0.05)], axis=-1)
    ds = np.linalg.norm(x[:, :, None, :] - POINT_SCENE[None, None], axis=-1) - (POINT_SCENE_RADIUS + radius)
    return np.minimum(d.min(axis=(1, 2)), ds.min(axis=(1, 2)))


def point_masses_reach(B: int, seed: int = 0, jitter: float = 0.3, offset: float = 0.5, margin: float = 0.1):
    """A solvable variant of the point-mass examples: the starts and scene of point_masses(B, seed, jitter), but every
    robot's goal lies `offset` from its own start in a uniformly drawn direction (PCG64(seed + 1)).  A direction is redrawn
    while the goal is closer than `margin` to contact with a scene sphere or another robot's goal.  (The examples' own swap
    goals put two robots' goals inside scene spheres, so no episode of them can succeed.)
    -> q0 (B,4,3), goals (B,4,2), scene (B,6,4)."""
    q0, _, scene = point_masses(B, seed, jitter)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    goals = np.zeros((B, 4, 2))
    todo = np.arange(B)
    while len(todo):
        ph = rng.uniform(0.0, 2.0 * math.pi, (len(todo), 4))
        g = q0[todo, :, 0:2] + offset * np.stack([np.cos(ph), np.sin(ph)], axis=-1)
        gq = np.concatenate([g, np.zeros(g.shape[:2] + (1,))], axis=-1)
        ok = point_start_clearance(gq) > margin
        goals[todo[ok]] = g[ok]
        todo = todo[~ok]
    return q0, goals, scene
