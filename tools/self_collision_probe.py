"""Cost of the self-collision leaves on the B200: executed action (R = 3, S = 64) and generic coupled rollout (R = 3,
H = 20) at 65 536 scenarios with 0 and with 4 pairs per robot, FP32 and FP64, and the B = 1 rollout latency with pairs
(generic kernel) against the cooperative kernel without.  CUDA events, median of 7 warm launches.

    python tools/self_collision_probe.py [--out profiles/r6_self_collision.md]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import multi_robot_fabrics_b200 as m  # noqa: E402
from multi_robot_fabrics_b200.api import Fabrics, to_soa  # noqa: E402

PAIRS4 = [(9, 2), (8, 3), (7, 4), (9, 1)]


def med_ms(fn, reps=7):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(min(ts)), float(max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--B", type=int, default=65536)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("self_collision_probe: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    R, B, S, H = 3, args.B, 64, 20
    rec = m.scenarios.generate(B, R, seed=1)
    rng = np.random.default_rng(0)
    rows = []
    fab = Fabrics(R, device=0)
    try:
        for dt, tdt in (("f32", torch.float32), ("f64", torch.float64)):
            d_rec = torch.from_numpy(to_soa(rec)).to("cuda:0", dtype=tdt)
            obst = torch.from_numpy(rng.uniform(-1, 1, size=(S, 10, R, B))).to("cuda:0", dtype=tdt)
            obst[:, 9] = 0.08
            act = torch.empty((7, R, B), dtype=tdt, device="cuda:0")
            for n in (0, 4):
                fab.set_self_collision([PAIRS4[:n]] * R if n else None, [[0.16] * n] * R if n else None)
                t = med_ms(lambda: fab.action_dev(d_rec, obst, action=act))
                rows.append((f"executed action, R=3, S=64, {dt}", n, t))
                t = med_ms(lambda: fab.rollout_dev(d_rec, H))
                rows.append((f"coupled rollout, R=3, H=20, {dt}", n, t))
        d1 = torch.from_numpy(to_soa(rec[:1])).to("cuda:0", dtype=torch.float32)
        fab.set_self_collision(None, None)
        rows.append(("B=1 rollout latency, R=3, H=20, f32 (cooperative kernel)", 0, med_ms(lambda: fab.rollout_dev(d1, H), 21)))
        fab.set_self_collision([PAIRS4] * R, [[0.16] * 4] * R)
        rows.append(("B=1 rollout latency, R=3, H=20, f32 (generic kernel)", 4, med_ms(lambda: fab.rollout_dev(d1, H), 21)))
    finally:
        fab.close()
    lines = [f"GPU: {smi}", "", "| workload | pairs/robot | median ms | min | max |", "|---|---|---|---|---|"]
    for name, n, (md, lo, hi) in rows:
        lines.append(f"| {name} | {n} | {md:.3f} | {lo:.3f} | {hi:.3f} |")
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
