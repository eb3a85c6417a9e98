#!/usr/bin/env python
"""bench.py -- fabric robot-steps/s of batched 3-Panda RF-CV rollouts (BASELINE.json's metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--horizon H] [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
              bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch of synthetic scenarios on every rank: the coupled RF-CV rollout
kernel (goal estimate + H horizon steps for 3 Pandas per scenario, FP32) followed by the post step
(mrf_rfcv_post_dev_f32, two kernels: the deadlock heuristic for every scenario the FP32 rollout decides safely + the list of
those in the guard band of a threshold; then their FP64 re-roll, each CTA followed by the heuristic for what it re-rolled;
both write the per-scenario result tensor avg_vel[R] + flag) and, for N > 1, the all_gather of that tensor -- no per-step
collective: four chunks of consecutive steps, each exchanged on a side stream under the rollouts that follow.  The steps
of a sweep are independent batches: the post step of step i runs on a side stream while the rollout streams already run
steps i+1, i+2 (eight output sets in flight; sharding.gather_into).  One
robot-step = one fabric action evaluation of one robot at one horizon step (FK/J/Jdot qdot, leaves, pullback, solve,
integrator update, avg-velocity accumulation).

  value     whole-job robot-steps/s with the scenario records already resident in HBM: CUDA events around EXACTLY K
            steps (first rollout launch -> last post step / gather complete), barrier + synchronize on both sides, max
            over ranks.  The steps rotate through 6 record sets (208 MB > the 126 MB L2), so no step finds its inputs
            in L2 and no flush sits inside the region.
  f64       the same sweep through the FP64 kernels (the parity path: 1e-9 relative against the oracle, checked on the
            timed batch), with its own roofline fraction against the FP64 FMA peak.
  e2e       the same metric AND THE SAME STEP (rollout + FP64 guard + deadlock heuristic) through the host-pointer C-ABI
            on page-locked buffers: mrf_rfcv_host_submit_f32 / mrf_rollout_host_wait, four batches in flight; the rollout
            kernel reads the compact records (per scenario and robot q, qdot, x_goal_0, weight_goal_0 + one shared record
            per batch) in the caller's order straight from host memory over PCIe, the post step runs on the device and
            the [R+1][B] result comes back.  Beside it, rollout only (what get_velocity_rollouts hands its Python caller:
            avg_vel / x_ee / goal_est written straight to host memory): compact-record pipeline, whole-record pipeline,
            and one blocking mrf_rollout_host_f32 call per step.
  roofline  the kernel is compute-bound on the FP32 CUDA-core pipe (arithmetic intensity > 200 FLOP/B, no tensor
            cores): achieved = robot-steps/s x F(S=16) = 13.4 kFLOP (SURVEY.md 8d) over the FMA peak measured in this
            run by the library's micro-benchmark (MEASURED_PEAKS.json holds HBM / bf16 peaks only); the HBM view is
            given beside it.  kernel_ms = CUDA events around every rollout launch of the timed region.
  cpu_baseline / --impl reference: the reference's dependencies (casadi / fabrics) are not installable offline, so the
            CPU arm is oracle O2 (closed-form C port, float64): ONE C call per step, goal estimate + rollout of every
            scenario inside one OpenMP loop on all host cores (thread count set explicitly, whatever OMP_NUM_THREADS
            the launcher exported), kind "port".
  --dump-outputs DIR  (--impl ours only) what the last timed step of `value` computed, device layout (scenario axis
            last) as float32 .npy: result (R+1,n) = avg_vel after the FP64 guard re-roll + deadlock flag, and the rollout's
            avg_vel (R,n), x_ee (R,3,n), goal_est (3,n), risk (R,n); scenario_index.npy holds the n positions in the step's
            batch that were written.  Written are the scenarios whose horizon the FP64 oracle finds calm (see calm(): the
            few that blow up have NaN or overflowed outputs in every implementation), all of them up to 64 MB, beyond
            that a fixed seeded sample; N > 1: one set per rank, suffix _rank<r>.  The timed batch itself is unchanged.
            Inputs and selection depend only on the arguments, so two builds run with the same arguments can be
            compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

N_ROBOTS = 3
FLOPS_PER_ROBOT_STEP = 5700 + 480 * 16      # SURVEY.md 8d / Appendix E, S = 8 (R-1) = 16 spheres
METRIC = "fabric robot-steps/sec (3 Panda RF-CV)"
UNIT = "robot-steps/s"
N_SETS = 6                                  # record sets the timed sweep rotates through (6 x 34.6 MB > L2)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="scenarios per GPU (weak scaling)")
    ap.add_argument("--horizon", type=int, default=20)
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="target duration of the CPU baseline sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-f64", action="store_true", help="skip the FP64 sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl ours: write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB "
                         "in all)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours only")
    return a


def config_dict(a):
    return {"workload": f"{a.batch} random 3-Panda scenarios per GPU x horizon {a.horizon}, RF-CV (goal estimate of "
                        f"robot 1, deadlock heuristic), joint-space coupled rollouts",
            "n_robots": N_ROBOTS, "horizon": a.horizon, "scenarios_per_gpu": a.batch, "spheres_seen_per_robot": 16,
            "parallelism": f"scenario-sharded x{a.gpus}",
            "l2": f"inputs larger than L2: the sweep rotates through {N_SETS} record sets ({N_SETS} x 34.6 MB at the default "
                  f"batch), no flush inside the timed region"}


# ------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle O2, the closed-form port) -- the only place bench.py executes oracle/.  It never loads the CUDA library.
# ------------------------------------------------------------------------------------------------------------------
def _scenarios():
    """Scenario generator without touching the CUDA library (importing the package does not dlopen it)."""
    import multi_robot_fabrics_b200 as m
    return m.scenarios


def calm(rec: np.ndarray, horizon: int) -> np.ndarray:
    """(B,) mask of the scenarios (B,R,44) whose FP64 horizon (oracle O2) stays calm: avg_vel finite and below 2 for
    every robot, the parity check's test.  The others blow up under explicit Euler near contact: velocities explode
    within a few steps, a joint is thrown past its limit, the fabric metric stops being positive definite and every
    implementation returns NaN or overflowed values (DESIGN.md section 2), so their outputs are not comparable."""
    from oracle import o2
    avg = o2.rollout_rfcv(o2.default_config(N_ROBOTS), rec.astype(np.float64), horizon, n_threads=o2.hw_threads())["avg_vel"]
    return np.isfinite(avg).all(axis=1) & (avg.max(axis=1) < 2.0)


def cpu_threads() -> int:
    from oracle import o2
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))     # undo a launcher's / our own per-rank pinning
    except OSError:
        pass
    return o2.hw_threads()


def cpu_step(cfg, rec, horizon: int, threads: int) -> float:
    """One step of the CPU path: RF-CV goal estimate + coupled rollout of every scenario, ONE OpenMP call."""
    from oracle import o2
    t0 = time.perf_counter()
    o2.rollout_rfcv(cfg, rec, horizon, est_robot=1, est_h=0.2, use_jqd=False, n_threads=threads)
    return time.perf_counter() - t0


def cpu_sample(horizon: int, target_s: float, seed: int = 0):
    from oracle import o2
    o2.build()
    cfg = o2.default_config(N_ROBOTS)
    threads = cpu_threads()
    gen = _scenarios().generate
    probe = gen(512, N_ROBOTS, seed=seed)
    cpu_step(cfg, probe[:64], horizon, threads)
    t = cpu_step(cfg, probe, horizon, threads)
    n = int(max(512, min(262144, 512 * target_s / max(t, 1e-6))))
    rec = gen(n, N_ROBOTS, seed=seed + 1)
    t = cpu_step(cfg, rec, horizon, threads)
    rs = n * N_ROBOTS * horizon / t
    return dict(value=rs, unit=UNIT, cores=threads, kind="port",
                sample=f"{n} scenarios x 3 Pandas x H{horizon} in {t:.2f} s, oracle O2 (closed-form C, float64, goal estimate + "
                       f"rollout in one OpenMP loop over scenarios, {threads} threads); the reference's casadi/fabrics wheels "
                       f"are not installable offline"), n, rec


def reference_arm(a):
    """--impl reference: the CPU implementation of the path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import o2
    per = max(1.0, min(8.0, 120.0 / max(1, a.steps + a.warmup)))
    base, n, rec = cpu_sample(a.horizon, per)
    cfg = o2.default_config(N_ROBOTS)
    threads = base["cores"]
    times = []
    for it in range(a.warmup + a.steps):
        dt = cpu_step(cfg, rec, a.horizon, threads)
        if it >= a.warmup:
            times.append(dt)
    total = sum(times)
    value = n * N_ROBOTS * a.horizon * len(times) / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(a),
            "cpu_baseline": dict(base, value=value,
                                 sample=f"each step = {n} scenarios x 3 Pandas x H{a.horizon} (a bounded sample of the config's "
                                        f"{a.batch}-scenario batch; throughput is per robot-step, so the sample size does not "
                                        f"enter the metric), oracle O2 port on {threads} host threads, one C call per step"),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region.  Polls NVML in-process every few ms (nvidia_ml_py)
    so that even a 20 ms region is sampled; falls back to an `nvidia-smi -lms` subprocess if NVML is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, device_index: int):
        self.idx = device_index
        self.rows = []          # (sm_mhz, power_w, reasons_mask)
        self.max_mhz = None
        self.proc = None
        self.nvml = None
        self.stop_flag = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((mhz, pw, mask))
            except Exception:
                pass
            time.sleep(0.004)

    def _read(self):
        names = {5: 0x8, 6: 0x40, 7: 0x20, 8: 0x4}
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                mask = 0
                for col, bit in names.items():
                    if r[col].lower().startswith("active"):
                        mask |= bit
                self.rows.append((float(r[1]), float(r[3]), mask))
                self.max_mhz = float(r[2])
            except Exception:
                continue

    def start(self):
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        self.stop_flag = True
        if self.nvml is not None:
            self.t.join(timeout=1.0)
        elif self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        else:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no NVML / nvidia-smi"]}
        sm = [r[0] for r in self.rows]
        pw = [r[1] for r in self.rows]
        mask = 0
        for r in self.rows:
            mask |= r[2]
        reasons = sorted(v for k, v in self.REASONS.items() if mask & k)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons,
                "source": "nvml in-process poll" if self.nvml is not None else "nvidia-smi -lms 20"}


def bind_to_gpu_socket(index: int) -> None:
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = {i for i in range(n) if (words[i // 64] >> (i % 64)) & 1} & os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def _sweep(fab, torch, dist, dev, world, recs, works, H, steps, warmup, with_risk):
    """K steps of the RF-CV sweep.  The steps are independent batches, so they are pipelined the way a production sweep
    runs them: rollouts alternate between TWO streams (the first wave of step i+1 fills the SMs that the last, partial
    wave of step i leaves idle: 2048 tiles on 592 CTA slots), the post step (+ gather) of every step runs on a third
    stream, NBUF output sets are in flight.  Returns total ms (events: before the first launch -> everything complete),
    per-launch rollout durations, buffers."""
    from multi_robot_fabrics_b200 import sharding
    _, R, B = recs[0].shape
    tdt = recs[0].dtype
    main = torch.cuda.current_stream(dev)
    NBUF = int(os.environ.get("MRF_BENCH_NBUF", "8"))
    NROLL = int(os.environ.get("MRF_BENCH_NROLL", "2"))
    roll = [torch.cuda.Stream(device=dev) for _ in range(NROLL)] if NROLL > 1 else [main]
    # the rollout kernels fill the register file of every SM, so the post step's two kernels run when rollout CTAs retire.
    # Measured (tools/sweep_probe.py): at normal priority with eight output sets in flight (the post chain of a step then
    # finishes in the tails of the next rollouts without ever holding one back) the step costs 1.008 ms, on high-priority
    # streams with four sets 1.018 ms
    # the post steps of consecutive batches overlap too (one FP64 re-roll tile has a latency of ~0.8 ms): one stream and
    # one scratch slot per output set
    NPOST = min(NBUF, 4, int(os.environ.get("MRF_BENCH_NPOST", "4")))
    sides = [torch.cuda.Stream(device=dev, priority=int(os.environ.get("MRF_BENCH_PRIO", "0"))) for _ in range(NPOST)]
    mk = lambda *shape, dtype=tdt: [torch.empty(shape, dtype=dtype, device=dev) for _ in range(NBUF)]
    avg, xee, gest, risk = mk(R, B), mk(R, 3, B), mk(3, B), mk(R, B)
    flag = mk(B, dtype=torch.int32)
    # per-scenario results (avg_vel[R] + flag) of EVERY timed step stay on the device; for N > 1 they are exchanged by ONE
    # all_gather after the last step, inside the timed region ("only a final NCCL gather", north star)
    results = torch.empty((steps, R + 1, B), dtype=tdt, device=dev)
    scratch = torch.empty((R + 1, B), dtype=tdt, device=dev)
    # N > 1: the result tensor is exchanged in a few chunks of consecutive steps, each all_gather issued on its own stream as
    # soon as the post steps of its chunk are enqueued, so that only the last chunk's transfer is not hidden behind the
    # rollouts that follow (one gather of all K steps after the sweep left 0.35 ms of NVLink time exposed at N = 8)
    n_chunks = max(1, min(int(os.environ.get("MRF_BENCH_GATHER_CHUNKS", "4")), steps)) if world > 1 else 0
    csz = -(-steps // n_chunks) if n_chunks else 0
    if csz > NBUF:              # a chunk's post_done events must all still belong to its own steps when it is issued
        csz = NBUF
    bounds = [(c0, min(c0 + csz, steps)) for c0 in range(0, steps, csz)] if n_chunks else []
    gathered = [torch.empty((world, c1 - c0, R + 1, B), dtype=tdt, device=dev) for c0, c1 in bounds] if world > 1 else None
    comm = torch.cuda.Stream(device=dev) if world > 1 else None
    # heuristic state per output set (concurrent post steps must not share the in/out state arrays)
    sm_state = [torch.zeros((R, B), dtype=torch.int32, device=dev) for _ in range(NBUF)]
    tstep = torch.full((B,), 100, dtype=torch.int32, device=dev)
    tdo = [torch.full((B,), 1000, dtype=torch.int32, device=dev) for _ in range(NBUF)]
    st_int = [torch.tensor([0, 1, 0, 1], dtype=torch.int32, device=dev).repeat_interleave(B).contiguous() for _ in range(NBUF)]
    st_goal = [torch.zeros((3, B), dtype=tdt, device=dev) for _ in range(NBUF)]
    roll_done = [torch.cuda.Event() for _ in range(NBUF)]
    post_done = [torch.cuda.Event() for _ in range(NBUF)]
    kev = []

    def step(i, timed):
        k, s_ = i % NBUF, i % len(recs)
        rs = roll[i % len(roll)]
        with torch.cuda.stream(rs):
            if i >= NBUF:
                rs.wait_event(post_done[k])        # the post step of step i-NBUF has consumed this output set
            if timed:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(rs)
            fab.rollout_dev(recs[s_], H, avg_vel=avg[k], x_ee=xee[k], goal_est=gest[k], risk=risk[k] if with_risk else None)
            if timed:
                e1.record(rs)
                kev.append((e0, e1))
            roll_done[k].record(rs)
        side = sides[k % NPOST]
        with torch.cuda.stream(side):
            side.wait_event(roll_done[k])
            fab.rfcv_post_dev(recs[s_], H, xee[k], works[s_], gest[k], avg[k], sm_state[k], tstep, tdo[k], st_int[k],
                              st_goal[k], risk=risk[k] if with_risk else None, flag=flag[k],
                              result=results[i - warmup] if timed else scratch, slot=k % NPOST)
            post_done[k].record(side)

    def join():
        for s_ in roll + sides:
            if s_ is not main:
                main.wait_stream(s_)

    for s_ in roll + sides:
        if s_ is not main:
            s_.wait_stream(main)
    for i in range(warmup):
        step(i, False)
    join()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(main)
    for s_ in roll + sides:
        if s_ is not main:
            s_.wait_event(t0)
    h0 = time.perf_counter()
    if comm is not None:
        comm.wait_event(t0)
    ci = 0
    for i in range(steps):
        step(warmup + i, True)
        if world > 1 and i + 1 == bounds[ci][1]:         # the chunk's last step is enqueued: exchange its results
            c0, c1 = bounds[ci]
            with torch.cuda.stream(comm):
                for j in range(c0, c1):
                    comm.wait_event(post_done[(warmup + j) % NBUF])
                sharding.gather_into(gathered[ci], results[c0:c1])   # the sweep's only exchange (per chunk of steps)
            ci += 1
    host_ms = (time.perf_counter() - h0) * 1e3
    join()
    if comm is not None:
        main.wait_stream(comm)
    t1.record(main)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    last = (warmup + steps - 1) % NBUF
    return dict(host_enqueue_ms=host_ms, total_ms=t0.elapsed_time(t1), kern_ms=[e0.elapsed_time(e1) for e0, e1 in kev],
                avg=avg[last], flag=flag[last], result=results[steps - 1], last_set=(warmup + steps - 1) % len(recs),
                x_ee=xee[last], goal_est=gest[last], risk=risk[last] if with_risk else None,
                gathered=gathered, rollout_streams=len(roll))


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays, keep, budget=DUMP_BYTES, suffix=""):
    """--dump-outputs: arrays (name -> device tensor, scenario axis last) at the scenario positions `keep` (ascending)
    as path/<name><suffix>.npy in float32, with scenario_index<suffix>.npy (float64) naming the positions written.
    All of `keep` when it fits in `budget` bytes, otherwise the same seeded sample of it from every array, so that runs
    with the same arguments write the same scenarios."""
    import torch
    per_scenario = 8 + sum(4 * t[..., 0].numel() for t in arrays.values())
    n = min(len(keep), (budget - 128 * (len(arrays) + 1)) // per_scenario)  # 128: the header of a .npy file
    idx = keep if n == len(keep) else np.sort(np.random.default_rng(0).choice(keep, size=n, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"scenario_index{suffix}.npy"), idx.astype(np.float64))
    for name, t in arrays.items():
        t = t.index_select(t.dim() - 1, torch.from_numpy(idx).to(t.device))
        np.save(os.path.join(path, f"{name}{suffix}.npy"), t.float().cpu().numpy())


def _isolated_kernel_ms(fab, torch, dev, recs, H, launches, with_risk=True):
    """The dominant kernel alone: `launches` rollout launches back to back on ONE stream, CUDA events around each
    (a second timed region over the same rotating record sets; nothing else runs on the GPU)."""
    _, R, B = recs[0].shape
    t = lambda *shape: torch.empty(shape, dtype=recs[0].dtype, device=dev)
    avg, xee, gest, risk = t(R, B), t(R, 3, B), t(3, B), t(R, B)
    ev = []
    for i in range(3 + launches):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fab.rollout_dev(recs[i % len(recs)], H, avg_vel=avg, x_ee=xee, goal_est=gest, risk=risk if with_risk else None)
        e1.record()
        if i >= 3:
            ev.append((e0, e1))
    torch.cuda.synchronize(dev)
    return statistics.mean(e0.elapsed_time(e1) for e0, e1 in ev)


def ours(a):
    import torch
    import torch.distributed as dist

    import __graft_entry__ as g
    import multi_robot_fabrics_b200 as m
    from multi_robot_fabrics_b200 import sharding
    from multi_robot_fabrics_b200.api import Fabrics, to_soa

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if rank == 0:
        g.build()
    # N > 1: keep each rank on the CPUs (and so, by first touch, the memory) of its GPU's socket -- the e2e kernel reads
    # the page-locked records over PCIe, and a buffer on the far socket costs every rank bandwidth.
    if world > 1:
        bind_to_gpu_socket(local)
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        dist.barrier()
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    R, B, H = N_ROBOTS, a.batch, a.horizon
    steps, warmup = a.steps, max(3, a.warmup)

    # ---- synthetic scenarios: B DISTINCT rejection-sampled scenarios, PCG64(seed = rank) ----
    rec_h64 = m.scenarios.generate(B, R, seed=rank)                                         # (B,R,44) float64
    rec_h = np.ascontiguousarray(rec_h64, dtype=np.float32)
    fab = Fabrics(R, device=local, estimate_goal=1)                                         # RF-CV
    base = torch.from_numpy(to_soa(rec_h)).to(dev)                                          # (44,R,B)
    recs = [base] + [torch.roll(base, shifts=(k * B) // N_SETS, dims=2).contiguous() for k in range(1, N_SETS)]
    works = [r.clone() for r in recs]     # the deadlock step mutates goals / weights in place, like the reference's lists

    # ---- timed region: value (device-resident inputs) ----
    peak32 = fab.handle.fma_peak_tflops(False)
    peak64 = fab.handle.fma_peak_tflops(True)
    sampler = ClockSampler(local)
    launches0 = fab.handle.launches
    torch.cuda.synchronize()
    sampler.start()
    if os.environ.get("MRF_BENCH_GUARD_BANDS"):      # diagnostics: override the guard tiers, e.g. "0,0,0,0,0,0"
        fab.set_guard(bands=[float(v) for v in os.environ["MRF_BENCH_GUARD_BANDS"].split(",")])
    sw = _sweep(fab, torch, dist, dev, world, recs, works, H, steps, warmup,
                with_risk=os.environ.get("MRF_BENCH_NORISK", "0") != "1")
    clocks = sampler.stop()
    if a.dump_outputs:
        outs = {"result": sw["result"], "avg_vel": sw["avg"], "x_ee": sw["x_ee"], "goal_est": sw["goal_est"]}
        if sw["risk"] is not None:
            outs["risk"] = sw["risk"]
        # the last step ran on a rolled record set: position i holds scenario (i - shift) % B of rec_h
        pos = np.arange(B)
        keep = pos[calm(rec_h, H)[(pos - (sw["last_set"] * B) // N_SETS) % B]]
        dump_outputs(a.dump_outputs, outs, keep, DUMP_BYTES // world, suffix=f"_rank{rank}" if world > 1 else "")
    launches = (fab.handle.launches - launches0) * steps // (steps + warmup)
    total_ms = torch.tensor([sw["total_ms"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_s = float(total_ms.item()) * 1e-3
    value = world * B * R * H * steps / total_s
    kernel_ms_overlapped = statistics.mean(sw["kern_ms"])      # per-launch duration while two launches share the GPU
    kernel_ms = _isolated_kernel_ms(fab, torch, dev, recs, H, steps)
    rerolled, overflow, _ = fab.guard_stats()
    guard = {"fp64_rerolled_per_step": rerolled / (steps + warmup), "overflow": overflow,
             "host_enqueue_ms_per_step": sw["host_enqueue_ms"] / steps}
    nonfinite = float((~torch.isfinite(sw["avg"])).any(dim=0).float().mean().item())

    # parity spot check of what was timed (oracle as the checker; not timed): avg_vel and deadlock flags of the last step
    parity = None
    if rank == 0:
        from oracle import o2
        from oracle.deadlock_ref import DeadlockOracle
        n_chk = min(B, 2048)
        shift = (sw["last_set"] * B) // N_SETS
        idx = (np.arange(n_chk) * (B // n_chk) + 1) % B                  # positions in the rolled set
        src = (idx - shift) % B                                         # ... are these scenarios of the generated batch
        ref = o2.rollout_rfcv(o2.default_config(R), rec_h[src].astype(np.float64), H, n_threads=cpu_threads())
        ti = torch.from_numpy(idx).to(dev)
        got = sw["result"][:, ti].T.double().cpu().numpy()               # (n, R+1)
        ok = np.isfinite(ref["avg_vel"]).all(axis=1) & (ref["avg_vel"].max(axis=1) < 2.0)
        parity = {"scenarios": int(ok.sum()), "max_abs_err_avg_vel": float(np.abs(got[:, :R] - ref["avg_vel"])[ok].max())}
        del ti

    # ---- FP64 sweep (the parity path) ----
    f64 = None
    if not a.no_f64:
        b64 = torch.from_numpy(to_soa(rec_h.astype(np.float64))).to(dev)
        recs64 = [b64, torch.roll(b64, shifts=B // 2, dims=2).contiguous()]               # 2 x 69 MB > L2
        works64 = [r.clone() for r in recs64]
        s64, w64 = max(3, steps // 4), 2
        sw64 = _sweep(fab, torch, dist, dev, world, recs64, works64, H, s64, w64, with_risk=False)
        t64 = torch.tensor([sw64["total_ms"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t64, op=dist.ReduceOp.MAX)
        k64 = _isolated_kernel_ms(fab, torch, dev, recs64, H, s64, with_risk=False)
        tf64 = B * R * H / (k64 * 1e-3) * FLOPS_PER_ROBOT_STEP / 1e12
        f64 = {"value": world * B * R * H * s64 / (float(t64.item()) * 1e-3), "unit": UNIT, "steps": s64,
               "ms_per_step": float(t64.item()) / s64, "kernel": "rollout_kernel<double>", "kernel_ms": k64,
               "roofline": {"bound": "fp64", "achieved": tf64, "peak": peak64, "unit": "TFLOP/s", "frac": tf64 / peak64}}
        if rank == 0:
            shift = (sw64["last_set"] * B) // 2
            src = (idx - shift) % B
            ref64 = o2.rollout_rfcv(o2.default_config(R), rec_h[src].astype(np.float64), H, n_threads=cpu_threads())
            got64 = sw64["result"][:, torch.from_numpy(idx).to(dev)].T.cpu().numpy()
            ok = np.isfinite(ref64["avg_vel"]).all(axis=1) & (ref64["avg_vel"].max(axis=1) < 2.0)
            den = np.maximum(np.abs(ref64["avg_vel"]), 1e-3)
            f64["parity_max_rel_err_avg_vel"] = float((np.abs(got64[:, :R] - ref64["avg_vel"]) / den)[ok].max())
            # deadlock flags of the FP32 sweep against the FP64 sweep on the same scenarios (both consumed the same records
            # and the same heuristic state history only if the step counts agree, so compare the velocity test only)
        del recs64, works64, b64

    # ---- N > 1: determinism of the sharded sweep (SURVEY 8e): shards of ONE global batch, gathered, equal the 1-GPU result ----
    determinism = None
    if world > 1:
        per = 2048
        glob = m.scenarios.generate(per * world, R, seed=4242).astype(np.float32)         # same batch on every rank
        def run(rec_np):
            n = rec_np.shape[0]
            d = torch.from_numpy(to_soa(rec_np)).to(dev)
            out = _sweep(fab, torch, dist, dev, 1, [d], [d.clone()], H, 1, 0, with_risk=True)
            return out["result"].clone()
        lo, hi = sharding.shard_range(per * world, rank, world)
        full = sharding.gather_results(run(glob[lo:hi]), per * world)
        if rank == 0:
            single = run(glob)
            determinism = {"global_batch": per * world, "shards": world,
                           "bitwise_equal_to_one_gpu": bool(torch.equal(full.view(torch.int32), single.view(torch.int32)))}

    # ---- e2e: host-pointer C-ABI, pinned host buffers, copies inside the timed region ----
    pin = lambda shape: torch.empty(shape, dtype=torch.float32).pin_memory().numpy()
    h_rec = pin((B, R, 44))
    h_rec[...] = rec_h
    out = {"avg_vel": pin((B, R)), "x_ee": pin((B, R, 3)), "goal_est": pin((B, 3))}
    for _ in range(3):
        fab.rollout_host(h_rec, H, dtype="f32", out=out)
    if world > 1:
        dist.barrier()
    e2e_steps = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fab.rollout_host(h_rec, H, dtype="f32", out=out)          # synchronous: returns after the results are in host memory
    e2e_total = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_total, op=dist.ReduceOp.MAX)
    e2e_sync = world * B * R * H * e2e_steps / float(e2e_total.item())
    # the sweep is a stream of INDEPENDENT batches: two-deep submit / wait pipeline over the same in-place path, two sets of
    # page-locked buffers; every step's records are read from host memory and its results land in host memory inside
    # the timed region (the PCIe reads of step i+1 overlap the horizons of step i)
    h_rec2 = pin((B, R, 44))
    h_rec2[...] = rec_h[::-1]                      # the second buffer set holds the scenarios in reverse order
    bufs = [(h_rec, out), (h_rec2, {"avg_vel": pin((B, R)), "x_ee": pin((B, R, 3)), "goal_est": pin((B, 3))})]
    pipe_steps = max(6, min(steps, 20))

    def pipeline(submit):
        for i in range(4):
            submit(i)
        fab.rollout_host_wait(all=True)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(pipe_steps):
            submit(i)
        fab.rollout_host_wait(all=True)
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * B * R * H * pipe_steps / float(t.item())

    e2e_full = pipeline(lambda i: fab.rollout_host_submit(bufs[i % 2][0], H, bufs[i % 2][1], dtype="f32"))
    full_avg = [bufs[0][1]["avg_vel"].copy(), bufs[1][1]["avg_vel"].copy()]
    # The scenarios differ in q, qdot, x_goal_0 and weight_goal_0 only -- the per-step entries of the reference's
    # inputs_action dict; every other argument (x_goal_1/2, weights 1/2, angle_goal_1, constraint_0, radii) is the same for
    # all scenarios, so a sweep can submit COMPACT records (18 of 44 scalars per robot) plus one shared (R,44) template per
    # batch: the same results with 41 % of the PCIe traffic, which is what bounds the step when eight GPUs share the host.
    assert np.all(rec_h[:, :, 18:] == rec_h[0:1, :, 18:])
    shared_tail = np.ascontiguousarray(rec_h[0])
    cbufs = []
    for hr, ho in bufs:
        cv = pin((B, R, 18))
        cv[...] = hr[:, :, :18]
        cbufs.append((cv, ho))
    e2e_rollout_compact = pipeline(lambda i: fab.rollout_host_submit(cbufs[i % 2][0], H, cbufs[i % 2][1], dtype="f32",
                                                                     shared=shared_tail))
    assert all(np.array_equal(full_avg[k].view(np.uint8), cbufs[k][1]["avg_vel"].view(np.uint8)) for k in range(2))
    assert np.array_equal(cbufs[0][1]["avg_vel"].view(np.uint8), np.ascontiguousarray(cbufs[1][1]["avg_vel"][::-1]).view(np.uint8))
    # THE SAME STEP AS `value`, end to end: rollout + FP64 guard + deadlock heuristic from the page-locked compact records,
    # only the [R+1][B] result (avg_vel rows + flag) travels back (mrf_rfcv_host_submit_f32, four batches in flight)
    h_res = [pin((R + 1, B)) for _ in range(4)]      # the RF-CV pipeline is four deep: four result buffers cycle
    e2e_value = pipeline(lambda i: fab.rfcv_host_submit(cbufs[i % 2][0], H, h_res[i % 4], shared=shared_tail, time_step=100))
    # same rollouts as the rollout-only pipeline, bit for bit, except the few scenarios the guard re-rolled in FP64
    chk = np.isfinite(full_avg[0]).all(axis=1)
    differ = int(((h_res[0][:R].T != full_avg[0]).any(axis=1) & chk).sum())
    assert differ <= 1024 and set(np.unique(h_res[0][R]).tolist()) <= {0.0, 1.0}, differ
    e2e_flags = int(h_res[0][R].sum())
    h2d = int(cbufs[0][0].nbytes + shared_tail.nbytes) * world      # whole job, like `value`
    d2h = int(h_res[0].nbytes) * world

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline ----
    rs_kernel = B * R * H / (kernel_ms * 1e-3)                       # one GPU, dominant kernel alone
    achieved_tf = rs_kernel * FLOPS_PER_ROBOT_STEP / 1e12
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    if os.path.exists(peaks_file):
        hbm_peak, hbm_src = float(json.load(open(peaks_file))["hbm_gbs"]), "MEASURED_PEAKS.json"
    alg_bytes = B * (R * 43 * 4 + (R + R + 3 * R + 3) * 4)        # records in; avg_vel + risk + x_ee + goal_est out
    traffic = None
    tfile = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tfile):
        traffic = json.load(open(tfile)).get("rollout_f32_bytes_per_launch")
    roofline = {"bound": "fp32", "achieved": achieved_tf, "peak": peak32, "unit": "TFLOP/s", "frac": achieved_tf / peak32,
                "traffic": traffic, "kernel": "rollout_kernel<float>", "kernel_ms": kernel_ms,
                "kernel_timing": "CUDA events around each of K launches issued back to back on one stream right after the "
                                 "sweep (the kernel alone, same rotating record sets); inside the sweep two launches overlap "
                                 "on two streams, so a launch there lasts kernel_ms_overlapped while the sweep completes one "
                                 "launch every ms_per_step",
                "kernel_ms_overlapped": kernel_ms_overlapped, "sweep_frac": value / world * FLOPS_PER_ROBOT_STEP / 1e12 / peak32,
                "flops_per_robot_step": FLOPS_PER_ROBOT_STEP,
                "peak_source": "FMA micro-benchmark (mrf_fma_peak) measured in this run; MEASURED_PEAKS.json has no "
                               "FP32/FP64 CUDA-core figure",
                "hbm": {"achieved": alg_bytes / (kernel_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes": alg_bytes,
                        "peak_source": hbm_src},
                "fp64_peak_tflops": peak64, "fp32_peak_tflops": peak32}

    # ---- single-rollout latency (3 Pandas, H = 20, one scenario) ----
    one = torch.from_numpy(to_soa(rec_h[:1])).to(dev)
    a1 = torch.empty((R, 1), dtype=torch.float32, device=dev)
    for _ in range(10):
        fab.rollout_dev(one, 20, avg_vel=a1)
    torch.cuda.synchronize()
    lat = []
    for _ in range(50):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fab.rollout_dev(one, 20, avg_vel=a1)
        e1.record()
        torch.cuda.synchronize()
        lat.append(e0.elapsed_time(e1) * 1e3)
    t0 = time.perf_counter()
    for _ in range(200):
        fab.rollout_dev(one, 20, avg_vel=a1)
    torch.cuda.synchronize()
    lat_wall = (time.perf_counter() - t0) / 200 * 1e6
    # one synchronous call from the caller with HOST pointers (pageable numpy in, numpy out): upload, launch(es), download
    one_h = np.ascontiguousarray(rec_h[:1])
    for _ in range(5):
        fab.rollout_host(one_h, 20, dtype="f32")
    lat_host = []
    for _ in range(50):
        t0 = time.perf_counter()
        fab.rollout_host(one_h, 20, dtype="f32")
        lat_host.append((time.perf_counter() - t0) * 1e6)

    cpu = None
    if not a.no_cpu and world == 1:                  # the CPU leg is reported at N = 1 only
        cpu, _, _ = cpu_sample(H, a.cpu_seconds)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": 1e3 * total_s / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_dict(a),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "deadlock_flags_raised": e2e_flags, "scenarios_carrying_fp64_values": differ,
                    "rollout_only_compact_value": e2e_rollout_compact, "rollout_only_full_records_value": e2e_full,
                    "rollout_only_synchronous_call_value": e2e_sync,
                    "timing": "host wall clock, max over ranks, page-locked buffers.  value = THE SAME STEP AS the device-timed "
                              "`value` (rollout + FP64 guard re-roll + deadlock heuristic) through mrf_rfcv_host_submit_f32 / "
                              "mrf_rollout_host_wait, four batches in flight: the rollout kernel reads each step's compact records "
                              "(per scenario and robot q, qdot, x_goal_0, weight_goal_0; the arguments shared by all scenarios once "
                              "per batch) in place over PCIe, the post step runs on the device, the [R+1][B] result (avg_vel rows + "
                              "deadlock flag) is copied back.  rollout_only_*: get_velocity_rollouts alone (avg_vel, x_ee, goal_est "
                              "written straight to host memory; 3.9 MB back per step) with compact records / whole 44-scalar "
                              "records / one blocking mrf_rollout_host_f32 call per step"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "f64": f64,
            "guard": guard, "nonfinite_scenario_fraction": nonfinite, "parity_spot_check": parity,
            "single_rollout_us": {"device_events_median": statistics.median(lat), "wall_back_to_back": lat_wall,
                                  "sync_host_call_wall_median": statistics.median(lat_host),
                                  "shape": "1 scenario x 3 Pandas x H20"},
            "determinism": determinism}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    a = parse()
    if a.impl == "reference":
        return reference_arm(a)
    return ours(a)


if __name__ == "__main__":
    sys.exit(main())
