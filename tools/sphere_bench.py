"""Cost and effect of the sphere obstacle penalty (gradient_mode 5 / 6) on one GPU.

Prints one JSON line: the card and its power limit (read in the same run);
  - solve: 65 536 cold-started problems at N 8, dt 0.1 (tolerance 1e-3), device events, median of
    the timed repetitions: mode 0 against mode 5 and mode 3 against mode 6 with 0, 8, 20 and 64
    spheres placed over the problems' region, and mode 2 on configs[2]'s map for scale;
  - configs4: BASELINE configs[4] (65 536 drones x 100 replans, N 8, dt 0.1, tolerance 1e-3) in the
    48-sphere world of tools/obstacle_loop_bench.py (256^3 grid at 0.2 m, collisions judged on it):
    mode 6 on the analytic spheres (weight 1000, margin 1 m) against mode 4 on the 1 m clearance
    field (weight 1e5); ms per 100 replans, the fraction of drones that collided, final distance;
  - plan_p50_ms: SE3MPCPlanner.plan() with avoid_obstacles=True and 0, 20 and 100 spheres (host
    clock around the call, which synchronises).

    python tools/sphere_bench.py [--reps 20]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from obstacle_loop_bench import card, drones, timed, world  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--problems", type=int, default=65536)
    args = ap.parse_args()
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    from dart_planner_b200.planner import BatchWorkspace

    if not torch.cuda.is_available():
        raise SystemExit("sphere_bench.py needs a CUDA device")
    out = {"card": card(), "solve_us": {}, "configs4": {}, "plan_p50_ms": {}}
    B, N, dt = args.problems, 8, 0.1
    rng = np.random.default_rng(1)
    p0 = rng.uniform(-10, 10, (B, 3))
    v0 = rng.uniform(-2, 2, (B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], 1)
    srng = np.random.default_rng(2)
    centers, radii = srng.uniform(-12, 12, (64, 3)) * [1, 1, 0.5] + [0, 0, 4], srng.uniform(0.8, 2.0, 64)

    def arm(mode, n=None, grid=None):
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3),
                         gradient_mode=mode, obstacle_free_level=0.5)
        ws = BatchWorkspace(pr, B, pinned=False)
        ws.set_inputs_device(p0, v0, goal)
        if n is not None:
            ws.set_spheres((centers[:n], radii[:n]), 0.5)
        if grid is not None:
            ws.set_map(None, penalty_grid=grid)
        return round(1e3 * timed(ws.solve_device, args.reps), 1)

    out["solve_us"]["mode0"] = arm(0)
    out["solve_us"]["mode3"] = arm(3)
    for n in (0, 8, 20, 64):
        out["solve_us"][f"mode5_n{n}"] = arm(5, n)
        out["solve_us"][f"mode6_n{n}"] = arm(6, n)
    g2 = dp.DenseOccupancyGrid((256, 256, 256), (-128, -128, -128), 0.2)
    g2.add_obstacles(np.random.default_rng(2).uniform(-15, 15, (20, 3)), np.random.default_rng(3).uniform(0.5, 2, 20))
    out["solve_us"]["mode2_configs2_map"] = arm(2, grid=g2)
    del g2

    occ = world()
    field = occ.clearance_field(1.0)
    D = 65536
    q0, qg = drones(occ, D)
    D = len(q0)
    wrng = np.random.default_rng(7)
    wc, wr = wrng.uniform(-15, 15, (48, 3)), wrng.uniform(0.8, 2.5, 48)
    for name, mode, kw, w in (("mode6_spheres_w1000_margin1", 6, dict(spheres=(wc, wr), sphere_margin=1.0), 1000.0),
                              ("mode4_clearance1m_w1e5", 4, dict(penalty_grid=field), 1e5)):
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3, obstacle_weight=w),
                         gradient_mode=mode)
        sim = ClosedLoopSim(pr, D, plant_dt=dt, collision_map=occ, **kw)
        sim.reset(q0, np.zeros_like(q0), qg)
        sim.run(2)
        sim.reset(q0, np.zeros_like(q0), qg)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sim.run(100)
        b.record()
        torch.cuda.synchronize()
        d = np.linalg.norm(sim.positions().cpu().numpy() - qg, axis=1)
        out["configs4"][name] = dict(ms_100_replans=round(a.elapsed_time(b), 2),
                                     collided=float((sim.first_collision().cpu().numpy() >= 0).mean()),
                                     dist_median=float(np.median(d)), dist_max=float(d.max()))
    out["configs4"]["drones"] = D

    cfg = dp.SE3MPCConfig(prediction_horizon=8, dt=0.1)
    state = dp.DroneState(timestamp=0.0, position=np.array([0.0, 0.0, 2.0]), velocity=np.zeros(3))
    prng = np.random.default_rng(9)
    for n in (0, 20, 100):
        pl = dp.SE3MPCPlanner(cfg, respect_config_dt=True, avoid_obstacles=True)
        pl.set_goal([8.0, 3.0, 4.0])
        for c, r in zip(prng.uniform(-10, 10, (n, 3)), prng.uniform(0.5, 1.5, n)):
            pl.add_obstacle(c, r)
        for _ in range(20):
            pl.plan(state)
        ts = []
        for _ in range(200):
            t0 = time.perf_counter()
            pl.plan(state)
            ts.append(1e3 * (time.perf_counter() - t0))
        out["plan_p50_ms"][f"n{n}"] = round(float(np.median(ts)), 4)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
