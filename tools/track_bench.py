"""Cost and effect of reference tracking (gradient_mode 7 / 8) on one GPU.

Prints one JSON line: the card and its power limit (read in the same run);
  - solve_us: cold-started batches of 4 096, 65 536 and 1 Mi problems at N 8, dt 0.1 (tolerance
    1e-3), device events, median of the timed repetitions: mode 3 (fly to the goal) against mode 7
    (track the straight line to the goal at 2 m/s), and mode 6 against mode 8 with 20 spheres over
    the problems' region; the mean iteration count of each arm beside it;
  - configs4: BASELINE configs[4]'s population (65 536 drones x 100 replans, N 8, dt 0.1, tolerance
    1e-3), each drone following its own circle (radius 2..5 m, 1.5..3 m/s) from a start on it with
    the circle's velocity: mode 7, and mode 8 in the 48-sphere world (weight 1000, margin 1 m);
    ms per 100 replans (device events around ClosedLoopSim.run), then in a second, recorded run the
    tracking error (distance to the current path sample over times 20..100, RMS and max).

    python tools/track_bench.py [--reps 20]
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from obstacle_loop_bench import card, timed  # noqa: E402


def circles(B, T, dt, seed=11):
    rng = np.random.default_rng(seed)
    c = np.concatenate([rng.uniform(-10, 10, (B, 2)), rng.uniform(3, 8, (B, 1))], 1)
    r = rng.uniform(2, 5, B)
    w = rng.uniform(1.5, 3.0, B) / r * rng.choice([-1.0, 1.0], B)
    th = rng.uniform(0, 2 * np.pi, B)[:, None] + w[:, None] * (np.arange(T) * dt)[None]
    P = np.stack([c[:, 0:1] + r[:, None] * np.cos(th), c[:, 1:2] + r[:, None] * np.sin(th),
                  np.repeat(c[:, 2:3], T, 1)], 2)
    V = np.stack([-(r * w)[:, None] * np.sin(th), (r * w)[:, None] * np.cos(th), np.zeros((B, T))], 2)
    return P, V


def lines(p0, goal, N, dt, speed=2.0):
    """straight line p0 -> goal at `speed`, held at the goal"""
    d = goal - p0
    L = np.linalg.norm(d, axis=1)
    u = d / np.maximum(L, 1e-300)[:, None]
    s = np.minimum(speed * dt * np.arange(N)[None], L[:, None])
    P = p0[:, None] + s[..., None] * u[:, None]
    V = np.where((s < L[:, None])[..., None], speed * u[:, None], 0.0)
    return P, V


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
        raise SystemExit("track_bench.py needs a CUDA device")
    out = {"card": card(), "solve_us": {}, "mean_nit": {}, "configs4": {}}
    N, dt = 8, 0.1
    srng = np.random.default_rng(2)
    centers, radii = srng.uniform(-12, 12, (20, 3)) * [1, 1, 0.5] + [0, 0, 4], srng.uniform(0.8, 2.0, 20)
    for B in (4096, 65536, 1 << 20):
        rng = np.random.default_rng(1)
        p0 = rng.uniform(-10, 10, (B, 3))
        v0 = rng.uniform(-2, 2, (B, 3))
        goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], 1)
        ref = lines(p0, goal, N, dt)
        for mode in (3, 7, 6, 8):
            pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3),
                             gradient_mode=mode)
            ws = BatchWorkspace(pr, B, pinned=False)
            ws.set_inputs_device(p0, v0, goal)
            if mode in (7, 8):
                ws.set_reference(*ref)
            if mode in (6, 8):
                ws.set_spheres((centers, radii), 0.5)
            key = f"B{B}_mode{mode}"
            out["solve_us"][key] = round(1e3 * timed(ws.solve_device, args.reps), 1)
            out["mean_nit"][key] = round(float(ws.solve_device().nit.float().mean().item()), 3)
            del ws
        torch.cuda.empty_cache()

    D, steps = 65536, 100
    P, V = circles(D, steps + N, dt)
    wrng = np.random.default_rng(7)
    wc, wr = wrng.uniform(-15, 15, (48, 3)), wrng.uniform(0.8, 2.5, 48)
    for name, mode, kw in (("mode7", 7, {}), ("mode8_sphere_world_margin1", 8, dict(spheres=(wc, wr), sphere_margin=1.0))):
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3, obstacle_weight=1000.0),
                         gradient_mode=mode)
        sim = ClosedLoopSim(pr, D, plant_dt=dt, reference_path=(P, V), **kw)
        sim.reset(P[:, 0], V[:, 0])
        sim.run(2)
        sim.reset(P[:, 0], V[:, 0])
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sim.run(steps)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        sim.reset(P[:, 0], V[:, 0])
        hist = sim.run(steps, record=True)
        j = np.arange(steps) + 1
        d = np.linalg.norm(hist - P[:, j].transpose(1, 0, 2), axis=2)[19:]
        out["configs4"][name] = dict(ms_100_replans=round(ms, 2), rms_error_m=float(np.sqrt((d ** 2).mean())),
                                     max_error_m=float(d.max()))
    out["configs4"]["drones"] = D
    print(json.dumps(out))


if __name__ == "__main__":
    main()
