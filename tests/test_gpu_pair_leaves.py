"""GPU tests of the shared robot-robot sphere leaves of the 3-robot FP32 throughput rollout: the pair path is taken per
scenario (every body radius equal) and per configuration (dynamic mode, jdot_sign == jdot_ref_sign); everything else
falls back to every robot evaluating its own leaves.  Each case is checked against the float64 oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200.api import Fabrics
from oracle import o2

R = 3


def _oracle(rec, N, **kw):
    qN, qdN, avg, _ = o2.rollout_jointspace(o2.default_config(R, **kw), np.ascontiguousarray(rec, dtype=np.float64), N)
    mx = np.abs(qdN).max(axis=(1, 2, 3))
    return qdN, avg, np.isfinite(mx) & (mx < 3.0)


def _roll(fab, rec, N):
    fab.handle.set_coop_max_batch(0)  # the throughput kernel at every batch size
    return fab.rollout_host(rec, N, dtype="f32", trajectories=True)


def _within_f32_tolerance(out, qdN, avg, ok):
    """The FP32 coverage tolerance of test_gpu_parity.py::test_rollout_f32_within_tolerance."""
    with np.errstate(invalid="ignore"):
        eqd = np.nan_to_num(np.abs(out["qdN"] - qdN).max(axis=(1, 2, 3)), nan=np.inf)[ok]
        ea = np.nan_to_num(np.abs(out["avg_vel"] - avg).max(axis=1), nan=np.inf)[ok]
    assert ok.sum() > 0.9 * len(ok)
    assert np.mean(eqd <= 2e-3) >= 0.99 and np.mean(ea <= 1e-3) >= 0.99
    assert np.median(eqd) < 5e-6


def test_unequal_radii_scenario_inside_a_uniform_tile(built):
    N, B, odd = 20, 64, 37
    rec = m.scenarios.generate(B, R, seed=211)
    fab = Fabrics(R, device=0)
    try:
        base = _roll(fab, rec, N)
        rec2 = rec.copy()
        rec2[odd, 1, o2.RB:o2.RB + 6] = [0.08, 0.07, 0.09, 0.06, 0.08, 0.1]
        out = _roll(fab, rec2, N)
        alone = _roll(fab, rec2[odd:odd + 1], N)
    finally:
        fab.close()
    keep = np.arange(B) != odd
    for k in ("qdN", "avg_vel"):
        assert np.array_equal(out[k][keep].view(np.uint8), base[k][keep].view(np.uint8)), k  # neighbours unchanged
        assert np.array_equal(out[k][odd].view(np.uint8), alone[k][0].view(np.uint8)), k      # as if rolled alone
    qdN, avg, ok = _oracle(rec2, N)
    assert ok[odd]
    assert np.abs(out["qdN"][odd] - qdN[odd]).max() < 2e-3
    _within_f32_tolerance(out, qdN, avg, ok)


@pytest.mark.parametrize("kw", [dict(jdot_sign=1.0, jdot_ref_sign=1.0),        # pair path, other sign convention
                                dict(static_or_dyn=0),                          # static fabrics: fall-back
                                dict(jdot_sign=1.0), dict(jdot_ref_sign=1.0)])  # mixed signs: fall-back
def test_pair_path_and_config_fallbacks_match_oracle(built, kw):
    N, B = 20, 256
    rec = m.scenarios.generate(B, R, seed=223)
    fab = Fabrics(R, device=0, **kw)
    try:
        out = _roll(fab, rec, N)
    finally:
        fab.close()
    _within_f32_tolerance(out, *_oracle(rec, N, **kw))
