"""CPU tests of the shared robot-robot sphere leaves of the 3-robot FP32 throughput rollout (mrf_device.cuh,
pair_leaves_eval / pair_leaves_rebuild): the host emulation walks the two stages with the CTA barrier between them.  In
FP64 the stage functions must reproduce the oracle to 1e-9 -- on the pair path and on the per-scenario fall-back."""
import ctypes as C
import os

import numpy as np
import pytest

import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200 import _lib
from oracle import o2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 3


class _Emul:
    """emul_pair_rollout_*: with the shared leaves (mrf_emul_pair.cpp); emul_rollout_*: the full leaf set (mrf_emul.cpp)"""

    def __init__(self):
        d = os.path.join(ROOT, "tests", "emul")
        self.pair, self.full = C.CDLL(os.path.join(d, "libmrf_emul_pair.so")), C.CDLL(os.path.join(d, "libmrf_emul.so"))


@pytest.fixture(scope="module")
def emul(built):
    return _Emul()


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _roll(L, fn, cfg, rec, N):
    B = rec.shape[0]
    o = dict(avg=np.zeros((B, R)), qN=np.zeros((B, R, N, 7)), qdN=np.zeros((B, R, N, 7)))
    rec = np.ascontiguousarray(rec, dtype=np.float64)
    if fn.startswith("emul_pair_"):
        rc = getattr(L.pair, fn)(C.byref(cfg), _dp(rec), N, _dp(o["avg"]), _dp(o["qN"]), _dp(o["qdN"]), C.c_longlong(B))
        assert rc == 0
    else:
        xee, goal = np.zeros((B, R, 3)), np.zeros((B, 3))
        getattr(L.full, fn)(C.byref(cfg), _dp(rec), N, _dp(o["avg"]), _dp(xee), _dp(goal), _dp(o["qN"]), _dp(o["qdN"]),
                            C.c_longlong(B))
    return o


def _oracle(rec, N, **kw):
    qN, qdN, avg, _ = o2.rollout_jointspace(o2.default_config(R, **kw), np.ascontiguousarray(rec, dtype=np.float64), N)
    mx = np.abs(qdN).max(axis=(1, 2, 3))
    return qdN, avg, np.isfinite(mx) & (mx < 3.0)


def _check(o, qdN, avg, ok, tol=1e-9):
    assert ok.sum() > 0.9 * len(ok)
    assert np.abs(o["qdN"] - qdN)[ok].max() / np.abs(qdN[ok]).max() < tol
    assert np.abs(o["avg"] - avg)[ok].max() < tol


@pytest.mark.parametrize("kw", [dict(), dict(jdot_sign=1.0, jdot_ref_sign=1.0)])
def test_pair_leaves_match_oracle(emul, kw):
    """The pair path itself (both sign conventions with sigma == aref): FP64 to 1e-9, FP32 within the FP32 tolerance."""
    N, B = 12, 40
    rec = m.scenarios.generate(B, R, seed=41)
    cfg = _lib.default_config(R, **kw)
    qdN, avg, ok = _oracle(rec, N, **kw)
    _check(_roll(emul, "emul_pair_rollout_f64", cfg, rec, N), qdN, avg, ok)
    o32 = _roll(emul, "emul_pair_rollout_f32", cfg, rec, N)
    assert np.abs(o32["qdN"] - qdN)[ok].max() < 2e-3
    # the shared leaves change the FP32 rounding only: same order as every robot evaluating all its leaves
    o32_all = _roll(emul, "emul_rollout_f32", cfg, rec, N)
    assert np.abs(o32["qdN"] - o32_all["qdN"])[ok].max() < 2e-3


@pytest.mark.parametrize("kw", [dict(static_or_dyn=0), dict(jdot_sign=1.0), dict(jdot_ref_sign=1.0)])
def test_pair_leaves_fall_back_by_config(emul, kw):
    """Static mode or sigma != aref: the leaves are not symmetric, every robot evaluates its own (FP64 to 1e-9)."""
    N, B = 8, 32
    rec = m.scenarios.generate(B, R, seed=43)
    cfg = _lib.default_config(R, **kw)
    qdN, avg, ok = _oracle(rec, N, **kw)
    o = _roll(emul, "emul_pair_rollout_f64", cfg, rec, N)
    _check(o, qdN, avg, ok)
    ref = _roll(emul, "emul_rollout_f64", cfg, rec, N)
    assert np.array_equal(o["qdN"], ref["qdN"])


def test_pair_leaves_fall_back_per_scenario(emul):
    """A scenario with unequal body radii inside a tile of uniform ones takes the full leaf set; its result is the
    oracle's and is bitwise what it gets rolled on its own; its neighbours are bitwise unchanged."""
    N, B, odd = 8, 32, 11
    rec = m.scenarios.generate(B, R, seed=47)
    cfg = _lib.default_config(R)
    base = {fn: _roll(emul, fn, cfg, rec, N) for fn in ("emul_pair_rollout_f64", "emul_pair_rollout_f32")}
    rec2 = rec.copy()
    rec2[odd, 1, o2.RB:o2.RB + 6] = [0.08, 0.07, 0.09, 0.06, 0.08, 0.1]
    qdN, avg, ok = _oracle(rec2, N)
    for fn, o in base.items():
        o2_ = _roll(emul, fn, cfg, rec2, N)
        keep = np.arange(B) != odd
        assert np.array_equal(o2_["qdN"][keep], o["qdN"][keep]), fn
        alone = _roll(emul, fn, cfg, rec2[odd:odd + 1], N)
        assert np.array_equal(o2_["qdN"][odd], alone["qdN"][0]), fn
    _check(_roll(emul, "emul_pair_rollout_f64", cfg, rec2, N), qdN, avg, ok)
