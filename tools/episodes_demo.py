"""Closed-loop sweep demo: success / deadlock statistics of MRDF vs RF vs RF-CV, with coupled joint-space rollouts and
with decoupled Cartesian rollouts (RF-Cart, RF-CV-Cart), on random 2- or 3-Panda reach tasks.
Environment: ED_R robots, ED_B scenarios, ED_T control steps, ED_N horizon, ED_NPL spheres per link, ED_MODES
comma-separated subset of the rows (default all), ED_PNP / ED_BLOCKS pick-and-place."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import multi_robot_fabrics_b200 as m
from multi_robot_fabrics_b200.episodes import BatchedEpisodes
R = int(os.environ.get("ED_R", 2)); B = int(os.environ.get("ED_B", 4096)); T = int(os.environ.get("ED_T", 400)); N = int(os.environ.get("ED_N", 10))
NPL = int(os.environ.get("ED_NPL", 1))
base = m.scenarios.generate(min(B, 4096), R, seed=5)
rec = np.tile(base, ((B + len(base) - 1) // len(base), 1, 1))[:B]
rec[:, :, 7:14] = 0.0
task = {}
if int(os.environ.get("ED_PNP", 0)):     # pick-and-place protocol instead of the reach task
    blocks, start = m.scenarios.pick_and_place_layout(rec, n_blocks=int(os.environ.get("ED_BLOCKS", 2)), seed=1)
    task = dict(blocks=blocks, start_goal=start)
MODES = (("MRDF", dict(rollout_fabrics=False)), ("RF", dict(rollout_fabrics=True, resolve_deadlocks=True)),
         ("RF-CV", dict(rollout_fabrics=True, resolve_deadlocks=True, estimate_goal=True)),
         ("RF-Cart", dict(rollout_fabrics=True, resolve_deadlocks=True, rollouts="cartesian")),
         ("RF-CV-Cart", dict(rollout_fabrics=True, resolve_deadlocks=True, estimate_goal=True, rollouts="cartesian")))
pick = os.environ.get("ED_MODES")
for name, kw in MODES:
    if pick and name not in pick.split(","):
        continue
    ep = BatchedEpisodes(rec, n_horizon=N, dtype="f32", n_obst_per_link=NPL, **kw, **task)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    res = ep.run(T).results()
    dt = time.perf_counter() - t0
    ok = res["success"]
    print(json.dumps(dict(mode=name, robots=R, scenarios=B, control_steps=T, horizon=N, n_per_link=NPL, wall_s=round(dt, 3),
                          episodes_per_s=round(B / dt, 1), control_steps_per_s=round(B * T / dt),
                          success_rate=float(ok.mean()), median_steps_to_success=float(np.median(res["steps_to_success"][ok])) if ok.any() else None,
                          scenarios_with_deadlock=float((res["deadlock_steps"] > 0).mean()),
                          min_clearance_p01=float(np.nanquantile(res["min_clearance"], 0.01)),
                          **({"blocks_picked_mean": float(res["blocks_picked"].mean())} if task else {}))))
