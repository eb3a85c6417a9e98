"""Closed-loop point-mass episodes (episodes.BatchedPointEpisodes): rate and task statistics of the static and dynamic
variants in FP32 and FP64 on two workloads over the examples' scene -- "swap", the examples' own start / goal swap
(scenarios.point_masses; two of its goals lie inside scene spheres, so no episode succeeds) and "reach", its solvable
variant with every goal 0.5 from its start (scenarios.point_masses_reach) -- beside the loop a user writes without it:
one mrf_point_action_dev call per robot per step plus torch staging and integration, on the same scenes.
Prints one JSON line per row (and appends them to --out).  Rates are robot-control-steps/s from CUDA events around the
launch, each timed --repeats times on a fresh episode (median, min, max); the algorithmic FLOP per robot-step is counted
below and set against mrf_fma_peak measured in the same run.

usage: point_episodes_demo.py [--B 65536] [--T 2000] [--T-loop 300] [--jitter 0.3] [--repeats 5] [--out results.jsonl]"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200.api import Fabrics
from multi_robot_fabrics_b200._lib import default_config
from multi_robot_fabrics_b200.episodes import BatchedPointEpisodes

# algorithmic FLOP of one robot-step, as point_action / point_episode_kernel are written: every +, -, *, sqrt, rsqrt,
# reciprocal, exp and tanh counts 1 (an FMA counts 2, as mrf_fma_peak counts it); comparisons and selects count 0.
LEAF = {"offsets + rho": 4, "n2, 1/n, n": 7, "x, 1/(n rho), 1/x": 7, "xdot, |w|^2, curvature": 12,
        "metric, energy and geometry forces": 13, "obstacle acceleration": 4, "forcing terms": 7,
        "pull-back into f, M, energy numerator": 21}
DYN_REL_VEL = 2                                   # w = qdot - qdot_j for a dynamic robot sphere
TAIL = {"goal offset and norm": 6, "attractor scalars": 10, "forced force": 10, "two 2x2 solves": 30,
        "qMq, |qdot|^2": 17, "energy and execution terms": 19, "damper": 19, "action": 6}
METRIC_SCENE, METRIC_ROBOT, REACH, INTEGRATE = 2, 5, 6, 12


def flop_per_robot_step(S, R, dynamic):
    leaf = sum(LEAF.values())
    return (S * leaf + (R - 1) * (leaf + (DYN_REL_VEL if dynamic else 0)) + sum(TAIL.values()) + S * METRIC_SCENE
            + (R - 1) * METRIC_ROBOT + REACH + INTEGRATE)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().split("\n")[0]
    return [s.strip() for s in out.split(",")]


def timed(fn):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    fn()
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) * 1e-3


def python_loop(q0, goals, scene, dynamic, T, tdt, fab):
    """What a user writes today: per step and robot, stage the record and obstacle tensors with torch, call
    mrf_point_action_dev, then integrate with torch (semi-implicit Euler).  -> seconds for T steps (CUDA events)."""
    dev = torch.device("cuda:0")
    B, R, _ = q0.shape
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev, dtype=tdt)
    q, qd = t(q0.transpose(1, 2, 0)), torch.zeros((R, 3, B), dtype=tdt, device=dev)       # (R,3,B)
    g = t(goals.transpose(1, 2, 0))
    sc = t(scene.transpose(1, 2, 0))                                                        # (S,4,B)
    wr = torch.tensor([1.0, 0.2], dtype=tdt, device=dev)[:, None].expand(2, B)
    rad = torch.full((R - 1, 1, B), 0.2, dtype=tdt, device=dev)
    zeros2 = torch.zeros((R - 1, 2, B), dtype=tdt, device=dev)
    dt = float(fab.cfg.dt)

    def step():
        acts = []
        for i in range(R):
            oth = [j for j in range(R) if j != i]
            rec = torch.cat([q[i], qd[i], g[i], wr]).contiguous()                           # (10,B)
            if dynamic:
                dyn = torch.cat([q[oth, 0:2], qd[oth, 0:2], zeros2, rad], dim=1).contiguous()
                a = fab.point_action_dev(rec, sc, dyn)
            else:
                stat = torch.cat([sc, torch.cat([q[oth], rad], dim=1)]).contiguous()
                a = fab.point_action_dev(rec, stat)
            acts.append(a)
        a = torch.stack(acts)
        a = torch.where(torch.isfinite(a).all(dim=1, keepdim=True), a, torch.zeros_like(a))
        qd.add_(dt * a)
        q.add_(dt * qd)

    step()                                                                                  # warm-up
    torch.cuda.synchronize()
    return timed(lambda: [step() for _ in range(T)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=65536)
    ap.add_argument("--T", type=int, default=2000)
    ap.add_argument("--T-loop", type=int, default=300)
    ap.add_argument("--jitter", type=float, default=0.3)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, plimit, maxclk = card()
    fab = Fabrics(config=default_config(1))
    peak = {"f32": fab.handle.fma_peak_tflops(False), "f64": fab.handle.fma_peak_tflops(True)}
    rows = []
    for workload in ("swap", "reach"):
        make = m.scenarios.point_masses if workload == "swap" else m.scenarios.point_masses_reach
        q0, goals, scene = make(a.B, seed=0, jitter=a.jitter)
        B, R, S = a.B, q0.shape[1], scene.shape[1]
        for dtype in ("f32", "f64"):
            for dynamic in (False, True):
                BatchedPointEpisodes(q0[:256], goals[:256], scene[:256], dynamic=dynamic, dtype=dtype).run(10).results()  # warm-up
                secs = []
                for _ in range(a.repeats):
                    ep = BatchedPointEpisodes(q0, goals, scene, dynamic=dynamic, dtype=dtype)
                    torch.cuda.synchronize()
                    secs.append(timed(lambda: ep.run(a.T)))
                res = ep.results()
                ok = res["success"]
                fl = flop_per_robot_step(S, R, dynamic)
                rates = sorted(B * R * a.T / s for s in secs)
                rate = float(np.median(rates))
                rows.append(dict(
                    row="episode kernel", workload=workload, variant="dynamic" if dynamic else "static", dtype=dtype,
                    scenarios=B, robots=R, control_steps=a.T, launches=1, repeats=a.repeats,
                    kernel_s_median=round(float(np.median(secs)), 5), robot_steps_per_s=float(f"{rate:.4g}"),
                    robot_steps_per_s_min=float(f"{rates[0]:.4g}"), robot_steps_per_s_max=float(f"{rates[-1]:.4g}"),
                    success_rate=float(ok.mean()),
                    median_steps_to_success=float(np.median(res["steps_to_success"][ok])) if ok.any() else None,
                    clear_robots_p01=float(np.quantile(res["min_clear_robots"], 0.01)),
                    clear_scene_p01=float(np.quantile(res["min_clear_scene"], 0.01)),
                    scenarios_with_nonfinite=float((res["nonfinite_steps"] > 0).mean()),
                    flop_per_robot_step=fl, achieved_tflops=round(rate * fl / 1e12, 3), fma_peak_tflops=round(peak[dtype], 2),
                    share_of_fma_peak=round(rate * fl / 1e12 / peak[dtype], 4)))
                print(json.dumps(rows[-1]), flush=True)
                if workload == "swap":
                    tdt = torch.float32 if dtype == "f32" else torch.float64
                    secs = sorted(python_loop(q0, goals, scene, dynamic, a.T_loop, tdt, fab) for _ in range(3))
                    rows.append(dict(row="python loop over mrf_point_action_dev", workload=workload,
                                     variant="dynamic" if dynamic else "static", dtype=dtype, scenarios=B, robots=R,
                                     control_steps=a.T_loop, repeats=3, wall_s_cuda_events_median=round(secs[1], 4),
                                     robot_steps_per_s=float(f"{B * R * a.T_loop / secs[1]:.4g}"),
                                     robot_steps_per_s_min=float(f"{B * R * a.T_loop / secs[2]:.4g}"),
                                     robot_steps_per_s_max=float(f"{B * R * a.T_loop / secs[0]:.4g}")))
                    print(json.dumps(rows[-1]), flush=True)
    meta = dict(row="card", name=name, power_limit=plimit, max_sm_clock=maxclk)
    print(json.dumps(meta))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            for r in rows + [meta]:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
