"""Cost and effect of the dynamics-consistent solve mode (gradient_mode 3 / 4) on one GPU.

Prints one JSON line: the card and its power limit (read in the same run); device-event times per
batched solve (after warm-up, median of the timed repetitions) in modes 0 / 1 / 3 / 4 at 4 096 problems
(one stream), 65 536 and 1 Mi problems; and BASELINE configs[4] (65 536 drones x 100 replans, dt 0.1,
N 8, warm starts) in modes 0 and 3 at convergence_tolerance 5e-2 and 1e-3: time, final distance to
goal (median / p99 / max) and the fraction of planned speeds (every step of the final plans) above
max_velocity, which mode 3 does not enforce.

    python tools/rollout_bench.py [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def inputs(B, seed):
    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-10, 10, (B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], axis=1)
    v0 = np.random.default_rng(seed + 40).uniform(-2, 2, (B, 3))
    return p0, v0, goal


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    from dart_planner_b200.planner import BatchWorkspace

    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench.py needs a CUDA device")
    out = {"card": card(), "solve_us": {}, "configs4": {}}
    grid = dp.DenseOccupancyGrid((256, 256, 256), (-128, -128, -128), 0.2)
    rng = np.random.default_rng(2)
    grid.add_obstacles(rng.uniform(-20, 20, (64, 3)), rng.uniform(0.5, 2.0, 64))
    cfg = dp.SE3MPCConfig(prediction_horizon=8, dt=0.1)
    for B in (4096, 65536, 1 << 20):
        p0, v0, goal = inputs(B, 4)
        for mode in (0, 1, 3, 4):
            ws = BatchWorkspace(make_params(cfg, gradient_mode=mode), B, pinned=False, outputs="solution")
            ws.set_inputs_device(p0, v0, goal)
            if mode in (2, 4):
                ws.set_map(grid, 1.0, 0.6)
            for _ in range(3):
                ws.solve_device()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
            for a, b in ev:
                a.record()
                ws.solve_device()
                b.record()
            torch.cuda.synchronize()
            out["solve_us"][f"mode{mode}_B{B}"] = round(float(np.median([a.elapsed_time(b) for a, b in ev])) * 1e3, 1)
            del ws
            torch.cuda.empty_cache()
    B, N, dt = 65536, 8, 0.1
    p0, v0, goal = inputs(B, 4)
    for mode in (0, 3):
        for tol in (5e-2, 1e-3):
            pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=tol), gradient_mode=mode)
            sim = ClosedLoopSim(pr, B, plant_dt=dt)
            sim.reset(p0, v0, goal)
            sim.run(2)                                   # warm-up (module load, first launches)
            sim.reset(p0, v0, goal)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sim.run(100)
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b)
            # speeds of the final plans: the rollout of every drone (mode 3) / the V rows (mode 0)
            V = sim.solution()[:, 3 * N:6 * N].reshape(B, N, 3)
            over = float((V.norm(dim=2) > pr.max_velocity).double().mean())
            d = np.linalg.norm(sim.positions().cpu().numpy() - goal, axis=1)
            out["configs4"][f"mode{mode}_tol{tol:g}"] = dict(
                ms_100_replans=round(ms, 2), dist_median=float(np.median(d)), dist_p99=float(np.percentile(d, 99)),
                dist_max=float(d.max()), frac_speed_over_max=over)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
