"""Cost and effect of the obstacle-aware closed loop on one GPU.

Prints one JSON line: the card and its power limit (read in the same run); device-event times
(after warm-up, median of the timed repetitions) of `signed_distance` and `clearance_field` on a
256^3 grid with float32 and float64 cells; and BASELINE configs[4] (65 536 drones x 100 replans,
N 8, dt 0.1, tolerance 1e-3, warm starts, every step's flown path checked against the map) in the
48-sphere world of tests/test_rollout_mode.py on a 256^3 grid at 0.2 m (the same spheres, twice the
resolution), with starts and goals at least 1.5 m from occupied cells, in four arms: mode 3 without
the map (the plain step), mode 3, mode 4 on the occupancy grid and mode 4 on the 1 m clearance
field (both at weight 1e5).  Per arm: ms per 100 replans, the fraction of drones whose path ever
entered an occupied cell, and the final distance to the goal (median / max).

    python tools/obstacle_loop_bench.py [--reps 20]
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


def world(dtype="float32"):
    import dart_planner_b200 as dp
    g = dp.DenseOccupancyGrid((256, 256, 256), (-128, -128, -128), 0.2, dtype=dtype)
    rng = np.random.default_rng(7)
    g.add_obstacles(rng.uniform(-15, 15, (48, 3)), rng.uniform(0.8, 2.5, 48))
    return g


def drones(grid, B, clearance=1.5, seed=4):
    phi = grid.signed_distance(0.6).cpu().numpy()
    org = np.array(grid.origin_voxel)

    def phi_at(p):
        k = np.floor(p / grid.resolution).astype(int) - org
        return phi[k[:, 2], k[:, 1], k[:, 0]]

    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-10, 10, (4 * B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (4 * B, 2)), rng.uniform(3, 8, (4 * B, 1))], 1)
    ok = (phi_at(p0) > clearance) & (phi_at(goal) > clearance)
    return p0[ok][:B], goal[ok][:B]


def timed(fn, reps):
    import torch
    for _ in range(3):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--drones", type=int, default=65536)
    args = ap.parse_args()
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params

    if not torch.cuda.is_available():
        raise SystemExit("obstacle_loop_bench.py needs a CUDA device")
    out = {"card": card(), "transform_ms": {}, "configs4": {}}
    for dtype in ("float32", "float64"):
        g = world(dtype)
        out["transform_ms"][f"signed_distance_{dtype}"] = round(timed(lambda: g.signed_distance(0.6), args.reps), 3)
        out["transform_ms"][f"clearance_field_{dtype}"] = round(timed(lambda: g.clearance_field(1.0), args.reps), 3)
        del g
    occ = world()
    field = occ.clearance_field(1.0)
    B, N, dt = args.drones, 8, 0.1
    p0, goal = drones(occ, B)
    B = len(p0)
    v0 = np.zeros_like(p0)
    arms = {"mode3_plain": (3, None, None), "mode3": (3, None, occ), "mode4_occupancy_w1e5": (4, occ, occ),
            "mode4_clearance1m_w1e5": (4, field, occ)}
    for name, (mode, pen, chk) in arms.items():
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3,
                                         obstacle_weight=1e5), gradient_mode=mode)
        sim = ClosedLoopSim(pr, B, plant_dt=dt, penalty_grid=pen, collision_map=chk)
        sim.reset(p0, v0, goal)
        sim.run(2)                                       # warm-up (module load, first launches)
        sim.reset(p0, v0, goal)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sim.run(100)
        b.record()
        torch.cuda.synchronize()
        d = np.linalg.norm(sim.positions().cpu().numpy() - goal, axis=1)
        out["configs4"][name] = dict(
            ms_100_replans=round(a.elapsed_time(b), 2),
            collided=None if chk is None else float((sim.first_collision().cpu().numpy() >= 0).mean()),
            dist_median=float(np.median(d)), dist_max=float(d.max()))
    out["configs4"]["drones"] = B
    print(json.dumps(out))


if __name__ == "__main__":
    main()
