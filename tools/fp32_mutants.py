"""Do the FP32 bounds bite?  Builds libmrf_b200.so variants with ONE arithmetic edit each in FP32-only code (a dropped
term, a swapped operand, a constant perturbed in its 4th-5th significant digit, a sphere weighted 0) and runs the
per-scenario FP32 tests (tests/test_gpu_fp32_paths.py) and the older FP32 tests against each with MRF_B200_LIB.

No edit changes an address computation, a loop bound, a barrier, a launch or a memory operation, so no variant can
fault or hang.

usage: python tools/fp32_mutants.py [--build-only | --run-only] [names...]
  builds go to build_ab/<name>.so (git-ignored; the copies of the sources to build_ab/<name>/), in parallel like
  tools/ab_build.sh; the run prints mutant -> caught by the older FP32 tests / caught by the new file (and the case that
  exceeds its bound by the largest factor).
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AB = os.path.join(ROOT, "build_ab")
DEVICE = "multi-robot-fabrics_b200/csrc/mrf_device.cuh"
KERNELS = "multi-robot-fabrics_b200/csrc/mrf_b200.cu"

# name -> (file, exact text (must occur once), replacement, what it breaks)
MUTANTS = {
    "leaf2_no_obst_acc": (
        DEVICE,
        "P2<T> fq = pfma(X, psplat(sigma), pfma(pmul(Mg, da), psplat(-aref), fl));",
        "P2<T> fq = pfma(X, psplat(sigma), fl);",
        "sphere_leaf2: the obstacle-acceleration term of the forcing dropped"),
    "leaf2_geom_const": (
        DEVICE,
        "P2<T> hh = pmul(ix4, psplat(T(-0.5)));\n    P2<T> fl = pmul(u1, hh);                                      // M h",
        "P2<T> hh = pmul(ix4, psplat(T(-0.50005)));\n    P2<T> fl = pmul(u1, hh);                                      // M h",
        "sphere_leaf2: geometry constant -0.5 perturbed in its 5th digit"),
    "obstmajor_rb34_swap": (
        DEVICE,
        "rbp[ps] = pmk(prm[(P_RB + 2 * ps) * NT + tid], prm[(P_RB + 2 * ps + 1) * NT + tid]);",
        "rbp[ps] = ps == 0 ? pmk(prm[(P_RB + 1) * NT + tid], prm[P_RB * NT + tid])\n"
        "                                : pmk(prm[(P_RB + 2 * ps) * NT + tid], prm[(P_RB + 2 * ps + 1) * NT + tid]);",
        "obstacle-major loop (executed action, Cartesian rollouts): link3 and link4 body radii swapped"),
    "pair_no_partner_energy": (
        KERNELS,
        "if (pair_on) pl.num += pls[2 * kPairSlots * NT + (r == 0 ? 2 : r - 1) * kTile + lane];",
        "if (pair_on) pl.num += T(0) * pls[2 * kPairSlots * NT + (r == 0 ? 2 : r - 1) * kTile + lane];",
        "shared robot-robot leaves: the partner's energy sum dropped"),
    "chol_pair_forced_pivot": (
        DEVICE,
        "P2<T> r = pmk(Mth<T>::rsqrt(-plo(s)), Mth<T>::rsqrt(-phi(s)));",
        "P2<T> r = pmk(Mth<T>::rsqrt(-plo(s)), Mth<T>::rsqrt(-(j == 5 ? plo(s) : phi(s))));",
        "chol_solve6n_pair: the forced half's last pivot taken from the geometry half"),
    "sincos_poly_const": (
        DEVICE,
        "-1.6666654611e-1f",
        "-1.6667654611e-1f",
        "FP32 sincos: cubic sine coefficient perturbed in its 5th digit"),
    "kin_acc_scale": (
        KERNELS,
        "aa = kin_load(kin, NT, tid, emap[l], 6) * cfg.sref;",
        "aa = kin_load(kin, NT, tid, emap[l], 6) * (sizeof(T) == 4 ? cfg.sref * T(1.0002) : cfg.sref);",
        "kinematics_kernel (FP32): the link accelerations scaled by 1.0002"),
    "cart_motion_k_minus_1": (
        KERNELS,
        "src.tk = T(k) * cfg.dt;",
        "src.tk = T(sizeof(T) == 4 ? k - 1 : k) * cfg.dt;",
        "Cartesian rollout (FP32): obstacles moved to step k-1 instead of k"),
    "ring_last_sphere_w0": (
        DEVICE,
        "                emit(cur, f);\n            }\n            cp_async_wait<0>();",
        "                if (sizeof(T) == 8 || o != S - 1 || (S & 3) == 0) emit(cur, f);\n            }\n"
        "            cp_async_wait<0>();",
        "cp.async ring (FP32): the last sphere of a list with S % 4 != 0 weighted 0"),
    "keepj8_from_link7": (
        DEVICE,
        "if (kKeepJ8 && e == kEgo - 1) have_j8 = true;",
        "if (kKeepJ8 && e >= kEgo - 2) have_j8 = true;",
        "kKeepJ8: the hand's attractor columns taken from link7 when link8 carries no leaves"),
    "risk_trace_yy": (
        DEVICE,
        "stiff_sum += (acc.A.xx + acc.A.yy) + acc.A.zz;",
        "stiff_sum += (acc.A.xx + acc.A.yy) + (sizeof(T) == 4 ? acc.A.yy : acc.A.zz);",
        "risk (FP32): trace(A_e) reads A_yy in place of A_zz"),
}

NEW_TESTS = ["tests/test_gpu_fp32_paths.py"]
OLD_TESTS = ["tests/test_gpu_parity.py", "tests/test_gpu_pair_leaves.py", "-k",
             "f32 or action or cartesian or static or subsets or degenerate or full_size or control_step or pair"]


def build(names):
    os.makedirs(AB, exist_ok=True)
    procs = []
    for name in names:
        path, old, new, _ = MUTANTS[name]
        tree = os.path.join(AB, name)
        shutil.rmtree(tree, ignore_errors=True)
        for d in ("multi-robot-fabrics_b200/csrc", "include"):
            shutil.copytree(os.path.join(ROOT, d), os.path.join(tree, d))
        src = open(os.path.join(tree, path)).read()
        n = src.count(old)
        if n != 1:
            raise SystemExit(f"{name}: the edit's text occurs {n} times in {path} (must be once)")
        open(os.path.join(tree, path), "w").write(src.replace(old, new))
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler",
               "-fPIC", "-shared", "-o", os.path.join(AB, f"{name}.so"),
               os.path.join(tree, "multi-robot-fabrics_b200/csrc/mrf_b200.cu")]
        log = open(os.path.join(AB, f"{name}.log"), "w")
        procs.append((name, subprocess.Popen(cmd, stdout=log, stderr=subprocess.STDOUT)))
    bad = [name for name, p in procs if p.wait() != 0]
    for name, _ in procs:
        print(("FAILED " if name in bad else "built ") + name)
    if bad:
        raise SystemExit(f"build failed: {bad} (see build_ab/<name>.log)")


def run_tests(lib, args, first_only):
    """-> (caught, the failure that exceeds its bound by the largest factor, or the first failing test)."""
    env = dict(os.environ, MRF_B200_LIB=lib)
    p = subprocess.run([sys.executable, "-m", "pytest", *(["-x"] if first_only else []), "-q", "-m", "gpu", "-p",
                        "no:cacheprovider", *args], cwd=ROOT, env=env, capture_output=True, text=True)
    out = p.stdout + p.stderr
    if p.returncode not in (0, 1):
        raise SystemExit(f"pytest exited with {p.returncode} under {lib}:\n{out[-3000:]}")
    hits = re.findall(r"AssertionError: (\S+: worst per-scenario error [^\n]*\(([0-9.e+]+)x\))", out)
    n_failed = re.search(r"(\d+) failed", out)
    if hits:
        worst = max(hits, key=lambda h: float(h[1]))[0]
        return p.returncode == 1, f"{n_failed.group(1) if n_failed else '?'} tests failed; largest: {worst}"
    f = re.search(r"^FAILED [^\n]*", out, re.M)
    return p.returncode == 1, f.group(0) if f else ""


def run(names):
    missing = [n for n in names if not os.path.exists(os.path.join(AB, f"{n}.so"))]
    if missing:
        raise SystemExit(f"not built: {missing} (python tools/fp32_mutants.py --build-only)")
    rows = []
    for name in names:
        lib = os.path.join(AB, f"{name}.so")
        old, _ = run_tests(lib, OLD_TESTS, True)
        new, why = run_tests(lib, NEW_TESTS, False)
        rows.append((name, old, new, why))
        print(f"{name:24s} old suite: {'caught' if old else 'MISSED':6s}  new file: {'caught' if new else 'MISSED':6s}  {why}",
              flush=True)
    print("\n| mutant | what it breaks | older FP32 tests | tests/test_gpu_fp32_paths.py |\n|---|---|---|---|")
    for name, old, new, why in rows:
        print(f"| {name} | {MUTANTS[name][3]} | {'caught' if old else 'missed'} | {'caught' if new else 'MISSED'} ({why}) |")
    return all(r[2] for r in rows)


def main(argv):
    names = [a for a in argv if not a.startswith("--")] or list(MUTANTS)
    unknown = [n for n in names if n not in MUTANTS]
    if unknown:
        raise SystemExit(f"unknown mutants {unknown}; known: {list(MUTANTS)}")
    if "--run-only" not in argv:
        build(names)
    if "--build-only" in argv:
        return 0
    return 0 if run(names) else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
