"""Cost of the differentiable solve's backward (dart_se3mpc_solve_vjp_batch) against its forward on one GPU.

Prints one JSON line: the card and its power limit (read in the same run), and for 4 096 and 65 536
problems at N 8, dt 0.1 (plan_batch's tolerance 5e-2, the benchmark's start distribution), modes 3 and
7 (the straight line to the goal at 2 m/s as the reference): device-event medians of the timed
repetitions of the forward (the solve, resident inputs) and of the VJP (upstream gradients on x and the
cost, every output written), their ratio, and the VJP's mean number of free thrust entries.

    python tools/vjp_bench.py [--reps 20]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from obstacle_loop_bench import card, timed  # noqa: E402
from track_bench import lines  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.config import make_params
    from dart_planner_b200.planner import BatchWorkspace

    if not torch.cuda.is_available():
        raise SystemExit("vjp_bench.py needs a CUDA device")
    out = {"card": card(), "forward_us": {}, "vjp_us": {}, "vjp_over_forward": {}, "mean_free": {}}
    N, dt = 8, 0.1
    L = _cabi.lib()
    for B in (4096, 65536):
        rng = np.random.default_rng(1)
        p0 = rng.uniform(-10, 10, (B, 3))
        v0 = rng.uniform(-2, 2, (B, 3))
        goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], 1)
        ref = lines(p0, goal, N, dt)
        for mode in (3, 7):
            pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt), gradient_mode=mode)
            ws = BatchWorkspace(pr, B, pinned=False)
            ws.set_inputs_device(p0, v0, goal)
            if mode == 7:
                ws.set_reference(*ref)
            ld = ws.ld
            x = ws.solve_device().out[:9 * N]
            f8 = dict(dtype=torch.float64, device="cuda")
            gx, gc = torch.randn((9 * N, ld), **f8), torch.randn(ld, **f8)
            g3 = [torch.empty((3, ld), **f8) for _ in range(3)]
            gref, gw = torch.empty((6 * N, ld), **f8), torch.empty((4, ld), **f8)
            st = torch.empty(ld, dtype=torch.int32, device="cuda")
            trk = _cabi.TrackRef(N, 0, ws.reference_dev.data_ptr()) if mode == 7 else None
            ip = ws.inp.data_ptr()

            def vjp():
                rc = L.dart_se3mpc_solve_vjp_batch(
                    C.byref(pr), B, ld, ip, ip + 3 * 8 * ld, ip + 6 * 8 * ld, None, x.data_ptr(),
                    None if trk is None else C.byref(trk), None, gx.data_ptr(), gc.data_ptr(),
                    *(t.data_ptr() for t in g3), gref.data_ptr(), gw.data_ptr(), st.data_ptr(),
                    torch.cuda.current_stream().cuda_stream)
                _cabi.check(rc, "dart_se3mpc_solve_vjp_batch")

            key = f"B{B}_mode{mode}"
            fwd = timed(ws.solve_device, args.reps)
            ws.solve_device()
            bwd = timed(vjp, args.reps)
            T = x[6 * N:, :B]
            lo = torch.tensor([-pr.tilt_thrust, -pr.tilt_thrust, pr.min_thrust], **f8).repeat(N)[:, None]
            hi = torch.tensor([pr.tilt_thrust, pr.tilt_thrust, pr.max_thrust], **f8).repeat(N)[:, None]
            out["forward_us"][key] = round(1e3 * fwd, 1)
            out["vjp_us"][key] = round(1e3 * bwd, 1)
            out["vjp_over_forward"][key] = round(bwd / fwd, 3)
            out["mean_free"][key] = round(float(((T != lo) & (T != hi)).sum(0).double().mean()), 2)
            out.setdefault("vjp_status_nonzero", {})[key] = int((st[:B] != 0).sum())
            del ws
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
