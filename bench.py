#!/usr/bin/env python
"""bench.py -- batched SE(3)-MPC solves/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch B]
                    [--dump-outputs DIR]

A "step" is one batched solve of the workload (BASELINE.json configs[1]: 4096 hover-to-goal
problems, seed 1, p0~U(-10,10)^3, v0=0, goal~U(-15,15)^2 x U(3,8), default airframe, N=8,
dt=0.1 from config/defaults.yaml) per GPU.  `value` times the solve kernel on HBM-resident
inputs; `e2e` times the same call from pinned HOST buffers (H2D + kernel + D2H of every
output) through the package's public BatchWorkspace API.  One JSON line on stdout (rank 0).

`--impl reference` times the CPU restatement of the reference path (oracle/, C, all host
threads) on the same workload; that and the `cpu_baseline` leg are the only places this file
touches oracle/.

`--dump-outputs DIR` writes what the last timed step of `value` (or of `--impl reference`)
returned to its caller as DIR/<field>.npy, so that two builds run with the same arguments can be
compared output for output (the inputs are seeded).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "batched SE(3)-MPC solves/sec"
UNIT = "solves/s"
L2_FLUSH_BYTES = 256 << 20
L2_BYTES = 126 << 20
E2E_DEPTH = 3
VALUE_DEPTH = int(os.environ.get("DART_BENCH_DEPTH", "4"))
DUMP_BYTES = 64 * 10 ** 6
DUMP_FIELDS = ("x", "cost", "nit", "nfev", "status", "task", "accelerations", "attitudes", "body_rates", "thrusts")


def workload_inputs(B, seed):
    """SURVEY.md 8(d) config 2 distribution (reference experiments/validation/benchmark_audit_improvements.py:292-302)."""
    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-10, 10, (B, 3))
    v0 = np.zeros((B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], axis=1)
    return p0, v0, goal


def alg_bytes_per_solve(N):
    """SURVEY.md 8(d): inputs 9 fp64 + outputs (19N+1) fp64 + 3 int32 (+1 int32 task code)."""
    return 8 * 9 + 8 * (19 * N + 1) + 4 * 4


def dump_outputs(out_dir, sol):
    """sol: the host result of one batched solve (HostSolution or oracle.BatchResult).  Writes each
    of DUMP_FIELDS as out_dir/<field>.npy in float64 (the int32 counters convert exactly) and
    index.npy, the problems the rows belong to: all of them, or a fixed seeded sample when the
    batch's outputs would exceed DUMP_BYTES."""
    B = len(sol.cost)
    per_problem = 8 * (1 + sum(np.asarray(getattr(sol, f))[0].size for f in DUMP_FIELDS))     # 1: index
    idx = np.arange(B)
    if B * per_problem > DUMP_BYTES:
        keep = (DUMP_BYTES - (64 << 10)) // per_problem          # 64 KiB left for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "index.npy"), idx.astype(np.float64))
    for f in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f + ".npy"), np.asarray(getattr(sol, f))[idx].astype(np.float64))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bind_to_gpu_numa(index):
    """Pin this rank to the CPUs NVML reports as local to its GPU, before any pinned buffer is
    allocated, so the end-to-end copies of the N ranks do not cross sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
        return True
    except Exception:
        return False


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.active = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._halt.is_set():
            if self.active.is_set():
                try:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.002)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def time_python_reference(args, cores):
    """The UNMODIFIED reference planner (baseline/_ref, staged by __graft_entry__.build()) on the
    same workload, one process per host core: baseline/run_reference.py in a subprocess."""
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "baseline", "run_reference.py"),
                            "--problems", str(args.batch), "--procs", str(cores), "--horizon", str(args.horizon),
                            "--dt", str(args.dt), "--seed", "1"], capture_output=True, text=True, timeout=600)
        out = json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:          # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}
    if "unavailable" in out:
        return out
    return {"value": out["value"], "unit": UNIT, "cores": out["procs"], "kind": "reference",
            "sample": f"one pass over the same {args.batch}-problem workload, unmodified reference "
                      "SE3MPCPlanner.plan_trajectory (pure Python + SciPy L-BFGS-B), one process per core",
            "single_solve_ms": out["single_solve_ms"], "cpu_model": out["cpu_model"],
            "per_core_solves_per_s": out["value"] / max(out["procs"], 1),
            "g2_check": {"thrust_z": out["g2_thrust_z"], "expected": out["g2_expected_thrust_z"]}}


def run_reference(args):
    """CPU arm: the oracle port of the reference path on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    B, N = args.batch, args.horizon
    cores = host_cores()
    params = oracle.make_params(horizon=N, dt=args.dt)
    p0, v0, goal = workload_inputs(B, 1)
    for _ in range(args.warmup):
        oracle.solve_batch(params, p0, v0, goal, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sol = oracle.solve_batch(params, p0, v0, goal, nthreads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sol)
    value = args.steps * B / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{args.steps} passes over the {B}-problem workload, oracle/ C port of "
                                   "se3_mpc_planner.py + L-BFGS-B, pthreads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        # the reference's own Python path on the same workload and cores, reported beside the port
        # (which is ~270x faster per core and is the arm the ratio is taken against)
        "cpu_baseline_reference": time_python_reference(args, cores),
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    return {"workload": f"{args.batch} batched hover-to-goal SE(3)-MPC solves per GPU (BASELINE configs[1]): "
                        f"seed 1, p0~U(-10,10)^3, v0=0, goal~U(-15,15)^2xU(3,8), default airframe m=1.5 kg",
            "batch_per_gpu": args.batch, "horizon": args.horizon, "dt": args.dt,
            "max_iterations": 15, "convergence_tolerance": 0.05, "gradient": "reference (:552-580)",
            "parallelism": f"dp{args.gpus} by problem index, replicated params, no collective in the solve",
            "steps_in_flight": VALUE_DEPTH,
            "l2": "value: inputs larger than L2 -- the launches cycle through resident input/output sets "
                  f"totalling > 2 x {L2_BYTES >> 20} MiB; per_launch_flushed and e2e_single_step: L2 flushed "
                  f"between timed steps ({L2_FLUSH_BYTES >> 20} MiB write); e2e: inputs and results live in "
                  "pinned host memory (nothing resident is re-read)"}


def sharded_config_legs(torch, dist, dp, params, world, rank, stream, dt):
    """BASELINE configs[3] and configs[4] on the `world` GPUs of this launch (all ranks call this):
    the global batch is cut by problem index, every GPU solves its resident slice, results return
    through ONE gather.  Device-timed (CUDA events on the launching stream around solve + gather +
    the copy into host memory on rank 0), max over ranks; strong scaling (the global size is fixed)."""
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.sharding import ShardedSolver, shard_range

    def max_over_ranks(ms):
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    out = {}
    # ---- configs[3]: 1 Mi Monte-Carlo initial states, one goal, seed 3 --------------------------
    Bg = 1 << 20
    rng = np.random.default_rng(3)
    p0 = rng.normal((0, 0, 2), 1.0, (Bg, 3))
    v0 = rng.normal(0, 0.5, (Bg, 3))
    goal = np.tile([10.0, 0.0, 5.0], (Bg, 1))
    lo, hi = shard_range(Bg, world, rank)
    # the replicated map: every rank holds the 256^3 grid of configs[2]; rank 0 rasterises the 64
    # spheres and ONE broadcast copies its cells into the other ranks' replicas (outside the timed
    # regions: the map is built once, the solves only read their local replica)
    from dart_planner_b200.sharding import replicate_map
    grid = dp.DenseOccupancyGrid((256, 256, 256), (-128, -128, -128), 0.2)
    if rank == 0:
        wr = np.random.default_rng(2)
        grid.add_obstacles(wr.uniform(-20, 20, (64, 3)), wr.uniform(0.5, 2.0, 64))
    torch.cuda.synchronize()
    replicate_map(grid, src=0)
    for outputs, transport in (("solution", "host_block"), ("solution", "gather"), ("all", "gather")):
        how = "written into a shared host block" if transport == "host_block" else "gathered to rank 0 host memory"
        key = f"configs[3] 1 Mi Monte-Carlo solves sharded by problem index, replicated map, {outputs} rows {how}"
        try:
            # (the shared host block either maps on every rank or raises on every rank: the ranks
            # stay in step and the leg is skipped together, e.g. on a box with a small /dev/shm)
            solver = ShardedSolver(params, outputs=outputs, transport=transport)
            solver.set_map(grid, 1.5, 0.6)      # fused is_trajectory_safe against the local replica
            solver.stage(p0[lo:hi], v0[lo:hi], goal[lo:hi], presliced=True, global_B=Bg)
            solver.run()                # maps the shared block
        except Exception as e:          # noqa: BLE001
            out[key] = {"unavailable": f"{type(e).__name__}: {e}"[:300], "n_gpus": world}
            continue
        solver.run()
        times = []
        sol = None
        for _ in range(5):
            sync_all()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            sol = solver.run()
            b.record(stream)
            torch.cuda.synchronize()
            times.append(max_over_ranks(a.elapsed_time(b)))
        ms = statistics.mean(times)
        leg = {"value": Bg / (ms * 1e-3), "unit": UNIT, "ms": ms, "n_gpus": world, "scaling": "strong",
               "row_bytes": None}
        if transport == "host_block":
            leg["transport"] = ("no collective: every rank's kernel writes the rows of its slice straight into ONE "
                                "page-locked host block shared by the ranks (its own PCIe link), a barrier ends the call")
        else:
            leg["transport"] = ("one NCCL gather of packed rows to rank 0 + one pinned copy per slice"
                                if world > 1 else "single GPU: one pinned copy of the packed rows")
        if rank == 0:
            leg["row_bytes"] = int((solver._block.stride if transport == "host_block" else solver._pinned.shape[1]) * 8)
            # bit-identity: rank 0 alone solves a sample spread over every shard
            idx = np.arange(0, Bg, 257)
            alone = dp.plan_batch(p0[idx], v0[idx], goal[idx], dp.SE3MPCConfig(prediction_horizon=int(params.horizon), dt=dt),
                                  grid=grid, safety_margin=1.5, collision_threshold=0.6, to_host=True)
            leg["identical_to_one_gpu_on_sample"] = bool(
                np.array_equal(sol.x[idx], alone.x) and np.array_equal(sol.cost[idx], alone.cost)
                and np.array_equal(sol.nfev[idx], alone.nfev) and np.array_equal(sol.status[idx], alone.status)
                and sol.first_hit is not None and np.array_equal(sol.first_hit[idx], alone.first_hit))
            leg["map"] = "256^3 grid, 64 spheres, replicated per GPU by one broadcast from rank 0; fused is_trajectory_safe"
            leg["unsafe_fraction"] = float((sol.first_hit >= 0).mean()) if sol.first_hit is not None else None
            if sol.first_hit is not None:      # first colliding step per trajectory (-1: safe)
                leg["first_hit_hist"] = {int(k): int(v) for k, v in zip(*np.unique(sol.first_hit, return_counts=True))}
            leg["sample"] = int(len(idx))
            leg["nit_hist"] = np.bincount(sol.nit, minlength=4).tolist()
        out[key] = leg
        if transport == "host_block":
            sync_all()
            solver._block.close()
        del solver, sol
    # ---- configs[4]: 65536 drones x 100 replans (10 s at 10 Hz), warm starts, resident state ----
    Bd = 65536
    a4, _, c4 = workload_inputs(Bd, 4)
    b4 = np.random.default_rng(44).uniform(-2, 2, (Bd, 3))
    lo, hi = shard_range(Bd, world, rank)
    sim = ClosedLoopSim(params, max(hi - lo, 1), plant_dt=dt)
    final = torch.empty((world * (Bd // world + 1), 3), dtype=torch.float64, device="cuda") if rank == 0 else None

    def closed_loop():
        sim.reset(a4[lo:hi], b4[lo:hi], c4[lo:hi])
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        sim.run(100, stream, track_counters=False)
        pos = sim.positions().contiguous()
        if world > 1:       # the only exchange: final positions to rank 0
            width = Bd // world + 1
            send = torch.zeros((width, 3), dtype=torch.float64, device="cuda")
            send[: hi - lo] = pos
            dist.gather(send, [final[r * width:(r + 1) * width] for r in range(world)] if rank == 0 else None, dst=0)
        b.record(stream)
        torch.cuda.synchronize()
        return max_over_ranks(a.elapsed_time(b)), pos

    closed_loop()
    cl_ms, pos = closed_loop()
    leg = {"value": Bd * 100 / (cl_ms * 1e-3), "unit": UNIT, "total_ms": cl_ms, "launches_per_gpu": 100 * sim.default_parts(),
           "sub_populations_in_flight": sim.default_parts(),
           "n_gpus": world, "scaling": "strong", "drones_per_gpu": int(hi - lo)}
    if rank == 0 and world > 1:
        # the first shard's final positions must equal a single-GPU run of the same drones
        ref = ClosedLoopSim(params, hi - lo, plant_dt=dt)
        ref.reset(a4[lo:hi], b4[lo:hi], c4[lo:hi])
        ref.run(100, stream, track_counters=False)
        leg["shard0_identical_to_standalone"] = bool(torch.equal(ref.positions(), pos)
                                                     and torch.equal(final[: hi - lo], pos))
    out["configs[4] closed loop: 65536 drones x 100 replans (10 s at 10 Hz), warm starts, resident state, sharded"] = leg
    return out


def time_steps(torch, fn, flush, steps, warmup, stream):
    """K timed steps, each bracketed by CUDA events on the launching stream, L2 flushed in
    between (outside the event pairs).  Returns summed milliseconds."""
    for _ in range(warmup):
        flush.zero_()
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        flush.zero_()
        a.record(stream)
        fn()
        b.record(stream)
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="problems per GPU per step")
    ap.add_argument("--horizon", type=int, default=8)
    ap.add_argument("--dt", type=float, default=0.1)
    ap.add_argument("--no-extras", action="store_true", help="skip sweep / latency / cpu baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (rank 0) as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: dart_planner_b200 has no CPU fallback")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    all_cpus = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_bound = bind_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import ctypes as C
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.config import make_params
    from dart_planner_b200.planner import BatchWorkspace

    L = _cabi.lib()
    cfg = dp.SE3MPCConfig(prediction_horizon=args.horizon, dt=args.dt)
    params = make_params(cfg)
    B, N = args.batch, args.horizon
    p0, v0, goal = workload_inputs(B, 1 + 1000 * rank)
    ws = BatchWorkspace(params, B, pinned=True, outputs="all")
    ws.set_inputs_device(p0, v0, goal)
    ws.stage_host_inputs(p0, v0, goal)
    stream = torch.cuda.current_stream()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()

    # ---- value: kernel on resident inputs ------------------------------------------------
    # The workload as a planning server sees it: a stream of batches.  K launches queued
    # between ONE pair of events on the launching stream, cycling through enough resident
    # input/output sets (each holding the named workload) that a set has left the L2 long before
    # it comes round again -- the timing rules' "inputs larger than L2" instead of a flush kernel
    # between launches, whose own tail and the event pair around every 30 us launch are what rank
    # jitter at N > 1 used to come from.  The per-launch, L2-flushed figure is reported beside it
    # (`per_launch_flushed`).
    per_set = B * (9 + 19 * N + 1) * 8 + 4 * B * 4
    nsets = max(4, -(-2 * L2_BYTES // per_set))
    ring = []
    for i in range(nsets):
        w = BatchWorkspace(params, B, pinned=False, outputs="all")
        w.set_inputs_device(p0, v0, goal)
        ring.append(w)
    def run_stream(depth, hint):
        """K steps, `depth` of them in flight (one stream each, round robin); one event pair around
        all of them on the launching stream.  Returns (milliseconds, launches, the last step's
        BatchSolution)."""
        streams = [stream] + [torch.cuda.Stream() for _ in range(depth - 1)]
        L.dart_se3mpc_set_inflight_hint(hint)
        try:
            for i in range(max(args.warmup, nsets)):
                ring[i % nsets].solve_device(streams[i % depth])
            barrier()
            n0 = L.dart_launch_count()
            # device-side wait the K launches are queued behind: long enough for the host to issue all
            # of them (~10 us each from Python), so that the device-timed region never waits for
            # the host -- one timed region of 200 steps is 3 ms, a hiccup of the issuing thread (GIL
            # hand-over to the clock sampler, a page fault) would otherwise show up as a slower GPU
            torch.cuda._sleep(int(min(max(2_000_000, args.steps * 30_000), 60_000_000)))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for st in streams[1:]:
                st.wait_event(e0)
            for i in range(args.steps):
                last = ring[i % nsets].solve_device(streams[i % depth])
            for st in streams[1:]:
                ev = torch.cuda.Event()
                ev.record(st)
                stream.wait_event(ev)
            e1.record(stream)
            torch.cuda.synchronize()
            return float(e0.elapsed_time(e1)), L.dart_launch_count() - n0, last
        finally:
            L.dart_se3mpc_set_inflight_hint(0)

    def max_over_ranks(x):
        tt = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # `value`: VALUE_DEPTH steps in flight -- the batches of a stream are independent, so a server
    # keeps several on the machine at once; the library is told (dart_se3mpc_set_inflight_hint) and
    # runs them in the throughput build.  `single_stream`: the same K steps strictly one after the
    # other on one stream (latency build).
    sampler.active.set()
    total_ms, launches, last = run_stream(VALUE_DEPTH, VALUE_DEPTH * B)
    sampler.active.clear()
    if args.dump_outputs and rank == 0:     # before single_stream overwrites the ring's results
        dump_outputs(args.dump_outputs, last.numpy())
    del last
    barrier()
    total_ms_max = max_over_ranks(total_ms)
    value = world * B * args.steps / (total_ms_max * 1e-3)
    sampler.active.set()
    single_ms, _, _ = run_stream(1, 0)
    sampler.active.clear()
    barrier()
    single_value = world * B * args.steps / (max_over_ranks(single_ms) * 1e-3)
    del ring
    # the same launch, one event pair per launch, L2 flushed in between (round-1 definition of `value`)
    barrier()
    sampler.active.set()
    ms = time_steps(torch, lambda: ws.solve_device(stream), flush, min(args.steps, 50), args.warmup, stream)
    sampler.active.clear()
    tf_ = torch.tensor([float(sum(ms))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tf_, op=dist.ReduceOp.MAX)
    flushed_value = world * B * len(ms) / (float(tf_.item()) * 1e-3)

    # ---- e2e: pinned host -> device -> solve -> pinned host -------------------------------
    barrier()
    sampler.active.set()
    # The kernel itself moves the data: it reads the pinned input block and writes one packed
    # result row per problem into pinned host memory over PCIe (zero-copy, BatchWorkspace.solve_rows).
    # The headline uses SOLUTION rows -- x, cost and the counters, i.e. what scipy's minimize hands
    # the reference planner (:256-268); the derived arrays of :582-654 are pure functions of the
    # thrust rows of x and HostSolution evaluates them on first access.  `e2e_full_rows` (below)
    # is the same call returning them from the device as well (twice the bytes).
    from dart_planner_b200.planner import HostSolution
    ws_e2e = BatchWorkspace(params, B, pinned=True, outputs="solution")
    use_rows = ws_e2e.rows_supported
    if use_rows:
        ws_e2e.stage_host_inputs(p0, v0, goal)
        e2e_call = lambda: ws_e2e.solve_rows(stream)
    else:
        e2e_call = lambda: ws.solve_staged(stream)
    ms_e2e = time_steps(torch, e2e_call, flush, min(args.steps, 50), args.warmup, stream)   # one step at a time
    # The headline: the same call as a stream of steps with several in flight (one workspace +
    # stream each, `solve_rows(wait=False)`): the row write-back of one step (2.6 MB over PCIe)
    # overlaps the solve of the next.  Every step reads its inputs from pinned host memory and
    # leaves its result rows in pinned host memory inside the timed region (start event before the
    # first launch, end event after the last stream has drained).  How many steps in flight pay
    # depends on the host: one GPU's link is busiest with three; eight GPUs writing into one host
    # memory system saturate it with fewer (more in flight only adds contention).  All depths up to
    # E2E_DEPTH are timed (K steps each, max over ranks) and the best is the headline; every
    # depth's figure is in `e2e.by_depth`.
    slots = [ws_e2e]
    streams = [stream]
    e2e_by_depth = {}
    if use_rows:
        for _ in range(E2E_DEPTH - 1):
            w = BatchWorkspace(params, B, pinned=True, outputs="solution")
            w.stage_host_inputs(p0, v0, goal)
            slots.append(w)
            streams.append(torch.cuda.Stream())

        def e2e_stream(depth):
            for i in range(max(args.warmup, 2 * depth)):
                slots[i % depth].solve_rows(streams[i % depth], wait=False)
            torch.cuda.synchronize()
            for w in slots[:depth]:
                w.h_rows.zero_()
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(2_000_000)
            s0.record(stream)
            for st in streams[1:depth]:
                st.wait_event(s0)
            for i in range(args.steps):
                slots[i % depth].solve_rows(streams[i % depth], wait=False)
            for st in streams[1:depth]:
                ev = torch.cuda.Event()
                ev.record(st)
                stream.wait_event(ev)
            s1.record(stream)
            torch.cuda.synchronize()
            tt = torch.tensor([float(s0.elapsed_time(s1))], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt.item())

        for depth in range(E2E_DEPTH, 0, -1):
            e2e_by_depth[depth] = e2e_stream(depth)
        e2e_depth = min(e2e_by_depth, key=e2e_by_depth.get)
        e2e_stream_ms = e2e_by_depth[e2e_depth]
        if e2e_depth != 1:
            e2e_stream(e2e_depth)      # leave every used slot holding a result of the chosen configuration
    else:
        e2e_depth = 1
        e2e_stream_ms = float(sum(ms_e2e)) * args.steps / len(ms_e2e)
    # what the host side can take: all ranks copy 64 MiB blocks device -> pinned host at once
    # (copy engine, 8 copies each), the ceiling for any result path into host memory on this box
    probe_d = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    probe_h = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
    probe_h.copy_(probe_d)
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record(stream)
    for _ in range(8):
        probe_h.copy_(probe_d, non_blocking=True)
    c1.record(stream)
    torch.cuda.synchronize()
    tt = torch.tensor([float(c0.elapsed_time(c1))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    d2h_gbs_aggregate = world * 8 * (64 << 20) / (float(tt.item()) * 1e-3) / 1e9
    del probe_d, probe_h
    dev = ws.solve_device(stream).numpy()
    if use_rows:    # what arrived in host memory is the resident solve's result, bit for bit
        got = HostSolution.from_solution_rows(N, ws_e2e.h_rows.numpy()[:B], params)
        e2e_checked = True
        for w in slots[:e2e_depth]:     # every slot's host block holds the resident solve's result
            got = HostSolution.from_solution_rows(N, w.h_rows.numpy()[:B], params)
            e2e_checked = e2e_checked and bool(
                np.array_equal(got.x, dev.x) and np.array_equal(got.cost, dev.cost)
                and np.array_equal(got.nfev, dev.nfev) and np.array_equal(got.status, dev.status)
                and np.allclose(got.attitudes, dev.attitudes, rtol=0, atol=1e-12)
                and np.allclose(got.body_rates, dev.body_rates, rtol=0, atol=1e-9)
                and np.allclose(got.thrusts, dev.thrusts, rtol=0, atol=1e-12))
    else:
        e2e_checked = bool(np.array_equal(ws.h_out.numpy()[: 9 * N, :B].T, dev.x))
    sampler.active.clear()
    barrier()
    t = torch.tensor([float(sum(ms_e2e))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (e2e_stream_ms * 1e-3)        # already the max over ranks
    e2e_single_value = world * B * len(ms_e2e) / (float(t[0].item()) * 1e-3)
    e2e_ms_per_step = e2e_stream_ms / args.steps
    if e2e_single_value > e2e_value:
        # launch -> wait -> next (the host in the loop) beats every streamed depth: the ranks' writes
        # into host memory collide less.  Seen on 8 GPUs; it is the same public call.
        e2e_value, e2e_depth, e2e_ms_per_step = e2e_single_value, 0, float(t[0].item()) / len(ms_e2e)
    del slots[1:]

    # ---- BASELINE configs[3] / configs[4] on all GPUs of this launch ----------------------------
    sharded = None
    if not args.no_extras:
        sampler.active.set()
        if world == 1:
            try:        # extras must not cost the headline line (one process: nobody waits for us)
                sharded = sharded_config_legs(torch, dist, dp, params, world, rank, stream, args.dt)
            except Exception as e:      # noqa: BLE001
                sharded = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
        else:
            sharded = sharded_config_legs(torch, dist, dp, params, world, rank, stream, args.dt)
        sampler.active.clear()

    if rank != 0:
        sampler.stop()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline of the solve kernel (rank 0) ----------------------------------------------
    hbm_peak, peak_src = load_peaks()
    kernel_ms = total_ms / args.steps      # rank 0's timed region of `value` per launch (launches overlap: the throughput-equivalent duration)
    ab = alg_bytes_per_solve(N) * B
    achieved_gbs = ab / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved_gbs / hbm_peak, "traffic": None, "peak_source": peak_src,
                "alg_bytes_per_solve": alg_bytes_per_solve(N), "kernel_ms": kernel_ms,
                "kernel": "se3mpc_solve_kernel"}
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        try:
            with open(traffic_file) as fh:
                tf = json.load(fh)
            ent = tf.get(f"B{B}_N{N}", {})
            roofline["traffic"] = ent.get("dram_bytes_per_launch")
            roofline["traffic_source"] = tf.get("source")
            # the steps in flight run in the throughput build: its per-solve instruction count is the
            # one ncu measured on the 65 536-problem launch of the same build
            thr = tf.get(f"B65536_N{N}", {})
            if VALUE_DEPTH > 1 and thr.get("warp_inst_per_solve"):
                ent = dict(thr, warp_inst_per_launch=thr["warp_inst_per_solve"] * B)
            if ent.get("warp_inst_per_launch"):
                # issue roofline: executed warp instructions per launch (ncu count of the same
                # launch) over the live kernel time, against 4 issue slots per SM per clock
                props = torch.cuda.get_device_properties(0)
                clk = (statistics.median(sampler.samples) if sampler.samples else (sampler.max_mhz or 1965)) * 1e6
                peak_issue = props.multi_processor_count * 4 * clk
                ach_issue = ent["warp_inst_per_launch"] / (kernel_ms * 1e-3)
                roofline["issue"] = {
                    "warp_inst_per_solve": ent["warp_inst_per_launch"] / B, "achieved": ach_issue / 1e9,
                    "peak": peak_issue / 1e9, "unit": "G warp-inst/s", "frac": ach_issue / peak_issue,
                    "ipc_per_sm": ach_issue / (props.multi_processor_count * clk),
                    "fp64_pipe_active_pct_under_ncu": ent.get("fp64_pipe_active_pct"),
                    "issue_active_pct_under_ncu": ent.get("issue_active_pct"),
                    "note": "the kernel is bound by instruction issue / dependent-chain latency, not by HBM or "
                            "FP64 flops: at this instruction count a full issue rate would be "
                            f"{peak_issue / (ent['warp_inst_per_launch'] / B) / 1e6:.0f} M solves/s per GPU "
                            "(DESIGN.md section 4, 'Where the ceiling is')"}
        except Exception:
            pass

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": ws.h2d_bytes,
                "d2h_bytes_per_step": ws_e2e.d2h_bytes_rows if use_rows else ws.d2h_bytes,
                "ms_per_step": e2e_ms_per_step, "steps_in_flight": e2e_depth,
                "by_depth": dict({"0 (launch, wait, next)": e2e_single_value},
                                 **{str(k): world * B * args.steps / (v * 1e-3) for k, v in sorted(e2e_by_depth.items())}),
                "host_d2h_ceiling": {"aggregate_gbs": d2h_gbs_aggregate, "per_gpu_gbs": d2h_gbs_aggregate / world,
                                     "as_solves_per_s": d2h_gbs_aggregate * 1e9 / (ws_e2e.d2h_bytes_rows / B) if use_rows else None,
                                     "note": "all ranks copying 64 MiB blocks device -> pinned host at once (copy engines)"},
                "api": ("dart_planner_b200.planner.BatchWorkspace(outputs='solution').solve_rows(wait=False) "
                        f"on {max(e2e_depth, 1)} workspaces / streams in rotation (pinned host buffers; the kernel reads "
                        "them and writes one row [x | cost | counters] per problem over PCIe itself, no separate "
                        "copies; derived arrays evaluated lazily on the host)")
                if use_rows else "dart_planner_b200.planner.BatchWorkspace.solve_staged (pinned host buffers)",
                "matches_resident_solve": e2e_checked},
        "e2e_single_step": {"value": e2e_single_value, "unit": UNIT, "ms_per_step": float(sum(ms_e2e)) / len(ms_e2e),
                            "note": "the same call, one step at a time (launch, wait, next): the latency of a step, "
                                    "not the throughput of a stream of steps"},
        "single_stream": {"value": single_value, "unit": UNIT, "ms_per_step": single_ms / args.steps,
                          "note": "the same K steps strictly one after the other on one stream (latency build)"},
        "per_launch_flushed": {"value": flushed_value, "unit": UNIT, "ms_per_step": float(sum(ms)) / len(ms),
                               "note": "one event pair per launch, L2 flushed before every launch (cold "
                                       "instruction and data caches): round 1's definition of `value`"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "host": {"numa_bound_to_gpu": bool(numa_bound), "cores_visible": len(all_cpus) if all_cpus else None},
    }
    if sharded is not None:
        line["sharded_configs"] = sharded
    info = [C.c_int32() for _ in range(5)]
    L.dart_se3mpc_set_inflight_hint(VALUE_DEPTH * B)      # the build the timed region of `value` ran
    rc_info = L.dart_se3mpc_kernel_info(C.byref(params), B, *[C.byref(i) for i in info])
    L.dart_se3mpc_set_inflight_hint(0)
    if rc_info == 0:
        line["kernel_info"] = {"lanes_per_problem": info[0].value, "block": info[1].value,
                               "grid": info[2].value, "smem_bytes": info[3].value,
                               "regs_per_thread": info[4].value}

    if world == 1 and not args.no_extras:
        # FP64 FMA peak probe (compute-roofline denominator)
        scratch = torch.zeros(8, dtype=torch.float64, device="cuda")
        th = C.c_int32()
        iters = 1 << 16
        for _ in range(2):
            L.dart_fp64_probe(iters, C.byref(th), scratch.data_ptr(), stream.cuda_stream)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.active.set()
        a.record(stream)
        L.dart_fp64_probe(iters, C.byref(th), scratch.data_ptr(), stream.cuda_stream)
        b.record(stream)
        torch.cuda.synchronize()
        sampler.active.clear()
        fp64_peak = th.value * 8.0 * iters * 2.0 / (a.elapsed_time(b) * 1e-3) / 1e12
        # CPU baseline + algorithmic flops from the instrumented oracle on the same batch
        import oracle
        if all_cpus is not None:
            os.sched_setaffinity(0, all_cpus)     # the CPU baseline uses every host core again
        cores = host_cores()
        oparams = oracle.make_params(horizon=N, dt=args.dt)
        r1 = oracle.solve_batch(oparams, p0, v0, goal, nthreads=cores)
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 10.0:
            oracle.solve_batch(oparams, p0, v0, goal, nthreads=cores)
            reps += 1
        cpu_dt = time.perf_counter() - t0
        line["cpu_baseline"] = {
            "value": reps * B / cpu_dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{reps} passes over the same {B}-problem workload (~10 s), oracle/ C port of "
                      "se3_mpc_planner.py + SciPy L-BFGS-B semantics, pthreads"}
        line["cpu_baseline_reference"] = time_python_reference(args, cores)
        flops_per_solve = r1.flops / B
        ach_tf = flops_per_solve * B / (kernel_ms * 1e-3) / 1e12
        roofline["fp64"] = {"achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                            "frac": ach_tf / fp64_peak, "alg_flops_per_solve": flops_per_solve,
                            "peak_source": "DFMA probe kernel measured in this run"}
        # parity of the timed configuration against the oracle (reported, not timed)
        sol = ws.solve_device(stream).numpy()
        relf = np.abs(sol.cost - r1.cost) / np.maximum(np.abs(r1.cost), 1.0)
        line["parity"] = {
            "vs": "oracle (pinned to the reference by tests/golden)",
            "max_rel_cost_err": float(relf.max()), "max_abs_x_err": float(np.abs(sol.x - r1.x).max()),
            "counter_agreement": float(((sol.nit == r1.nit) & (sol.nfev == r1.nfev) & (sol.status == r1.status)).mean()),
            "nit_hist": np.bincount(sol.nit, minlength=4).tolist()}
        # larger batches (same distribution): throughput once the machine is full
        sweep = {}
        for Bs in (65536, 1 << 20):
            w2 = BatchWorkspace(params, Bs, pinned=True, outputs="all")
            a0, b0, c0 = workload_inputs(Bs, 2)
            w2.set_inputs_device(a0, b0, c0)
            w2.stage_host_inputs(a0, b0, c0)
            sampler.active.set()
            m1 = time_steps(torch, lambda: w2.solve_device(stream), flush, 10, 3, stream)
            m2 = time_steps(torch, lambda: w2.solve_staged(stream), flush, 5, 3, stream)
            w2s = BatchWorkspace(params, Bs, pinned=True, outputs="solution")
            w2s.stage_host_inputs(a0, b0, c0)
            m3 = time_steps(torch, lambda: w2s.solve_rows(stream), flush, 5, 3, stream)
            # rows come from the latency build, the resident solve at this size from the throughput
            # build: same counters, x equal to rounding (a few products are contracted differently
            # in the exact-size code copies; tools/variant_diff.py) -- compared as such
            hs = HostSolution.from_solution_rows(N, w2s.h_rows.numpy()[:Bs], params)
            dv = w2.solve_device(stream).numpy()
            rows_ok = bool(np.array_equal(hs.nfev[::97], dv.nfev[::97]) and np.array_equal(hs.status[::97], dv.status[::97])
                           and float(np.abs(hs.x[::97] - dv.x[::97]).max()) < 1e-12)
            del w2s
            sampler.active.clear()
            k_ms = statistics.mean(m1)
            sweep[f"B{Bs}"] = {"value": Bs / (k_ms * 1e-3), "kernel_ms": k_ms,
                               "hbm_frac": alg_bytes_per_solve(N) * Bs / (k_ms * 1e-3) / 1e9 / hbm_peak,
                               "fp64_frac": flops_per_solve * Bs / (k_ms * 1e-3) / 1e12 / fp64_peak,
                               "e2e_value": Bs / (statistics.mean(m3) * 1e-3),
                               "e2e_matches_resident_solve": rows_ok,
                               "e2e_full_soa_copies_value": Bs / (statistics.mean(m2) * 1e-3)}
            del w2
        line["sweep"] = sweep
        # end to end with FULL rows: the derived arrays (acceleration, attitude, body rate, thrust
        # magnitude) computed on the device and transferred too -- 1 280 B instead of 640 B per solve
        if ws.rows_supported:
            sampler.active.set()
            mf = time_steps(torch, lambda: ws.solve_rows(stream), flush, 50, 5, stream)
            sampler.active.clear()
            gf = HostSolution.from_packed_rows(N, ws.h_rows.numpy()[:B])
            line["e2e_full_rows"] = {
                "value": B / (statistics.mean(mf) * 1e-3), "unit": UNIT, "ms_per_step": statistics.mean(mf),
                "h2d_bytes_per_step": ws.h2d_bytes, "d2h_bytes_per_step": ws.d2h_bytes_rows,
                "matches_resident_solve": bool(np.array_equal(gf.x, dev.x) and np.array_equal(gf.body_rates, dev.body_rates)
                                               and np.array_equal(gf.nfev, dev.nfev)),
                "api": "BatchWorkspace(outputs='all').solve_rows"}
        # end to end with controls rows (thrust vectors + cost + counters only: what a server that
        # forwards thrust commands sends back)
        wc = BatchWorkspace(params, B, pinned=True, outputs="controls")
        if wc.rows_supported:
            wc.stage_host_inputs(p0, v0, goal)
            sampler.active.set()
            mc = time_steps(torch, lambda: wc.solve_rows(stream), flush, 50, 5, stream)
            sampler.active.clear()
            from dart_planner_b200.planner import HostSolution as _HS
            gc = _HS.from_control_rows(N, wc.h_rows.numpy()[:B])
            line["e2e_controls_rows"] = {
                "value": B / (statistics.mean(mc) * 1e-3), "unit": UNIT, "ms_per_step": statistics.mean(mc),
                "h2d_bytes_per_step": wc.h2d_bytes, "d2h_bytes_per_step": wc.d2h_bytes_rows,
                "matches_resident_solve": bool(np.array_equal(gc.thrust_vectors, dev.thrust_vectors)
                                               and np.array_equal(gc.nfev, dev.nfev)),
                "api": "BatchWorkspace(outputs='controls').solve_rows"}
        del wc
        # the other BASELINE configs, timed once each (kernel-only, resident inputs); their
        # parity lives in tests/test_gpu_config3.py and tests/test_gpu_closed_loop.py
        others = {}
        rng = np.random.default_rng(2)
        grid = dp.DenseOccupancyGrid((256, 256, 256), (-128, -128, -128), 0.2)
        grid.add_obstacles(rng.uniform(-20, 20, (64, 3)), rng.uniform(0.5, 2.0, 64))
        Bs = 65536
        a0, b0, c0 = workload_inputs(Bs, 2)
        b0 = np.random.default_rng(22).uniform(-2, 2, (Bs, 3))
        w3 = BatchWorkspace(params, Bs, pinned=False, outputs="all")
        w3.set_inputs_device(a0, b0, c0)
        w3.set_map(grid, 1.5, 0.6)
        m3 = time_steps(torch, lambda: w3.solve_device(stream), flush, 10, 3, stream)
        unsafe = float((w3.hit[:Bs] >= 0).float().mean().item())
        others["configs[2] 65536 solves + fused is_trajectory_safe on a 256^3 grid"] = {
            "value": Bs / (statistics.mean(m3) * 1e-3), "unit": UNIT, "kernel_ms": statistics.mean(m3),
            "unsafe_fraction": unsafe}
        p2 = make_params(cfg, gradient_mode=2)
        w3p = BatchWorkspace(p2, Bs, pinned=False, outputs="all")
        w3p.set_inputs_device(a0, b0, c0)
        w3p.set_map(grid, 1.5, 0.6)
        m3p = time_steps(torch, lambda: w3p.solve_device(stream), flush, 10, 3, stream)
        others["configs[2] same with the occupancy-grid obstacle penalty in the solve (extension, self-oracle)"] = {
            "value": Bs / (statistics.mean(m3p) * 1e-3), "unit": UNIT, "kernel_ms": statistics.mean(m3p),
            "unsafe_fraction": float((w3p.hit[:Bs] >= 0).float().mean().item())}
        del w3, w3p
        from dart_planner_b200.closed_loop import ClosedLoopSim
        sim = ClosedLoopSim(params, Bs, plant_dt=args.dt)
        a4, _, c4 = workload_inputs(Bs, 4)
        b4 = np.random.default_rng(44).uniform(-2, 2, (Bs, 3))
        sim.reset(a4, b4, c4)
        sim.run(3, stream, track_counters=False)
        sim.reset(a4, b4, c4)
        torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record(stream)
        sim.run(100, stream, track_counters=False)
        eb.record(stream)
        torch.cuda.synchronize()
        cl_ms = ea.elapsed_time(eb)
        others["configs[4] closed loop: 65536 drones x 100 replans (10 s at 10 Hz), warm starts, resident state"] = {
            "value": Bs * 100 / (cl_ms * 1e-3), "unit": UNIT, "total_ms": cl_ms,
            "launches": 100 * sim.default_parts(), "sub_populations_in_flight": sim.default_parts()}
        # mapper: one LiDAR-like scan (update_map) and the batched queries, the HBM/L2-bound side
        rngm = np.random.default_rng(3)
        R = 200_000
        sensors = rngm.uniform(-10, 10, (8, 3))
        rpos = sensors[rngm.integers(0, 8, R)]
        rdir = rngm.normal(0, 1, (R, 3))
        rhit = rngm.uniform(0.5, 30.0, R)
        rhit[rngm.random(R) < 0.25] = np.nan
        g2 = dp.DenseOccupancyGrid((256, 256, 256), (-128, -128, -128), 0.2, max_range=25.0)
        g2.update_map(rpos, rdir, rhit, 30.0)                       # warm-up (allocates the counters)
        torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record(stream)
        upd = g2.update_map(rpos, rdir, rhit, 30.0)
        eb.record(stream)
        torch.cuda.synchronize()
        um_ms = ea.elapsed_time(eb)
        ncell = 256 ** 3
        others["mapper update_map: 200k rays into a 256^3 grid (ray walk + Bayes apply, incl. host staging of the scan)"] = {
            "value": R / (um_ms * 1e-3), "unit": "rays/s", "total_ms": um_ms, "voxel_visits": upd["updated_voxels"],
            "apply_pass_min_bytes": ncell * 12}
        # the same scan from device-resident point clouds through the no-sync entry (two launches,
        # nothing read back): what a scan-rate caller pays
        d_start = torch.as_tensor(rpos.T.copy(), device="cuda")
        d_dir = torch.as_tensor(rdir.T.copy(), device="cuda")
        d_hit = torch.as_tensor(rhit, device="cuda")
        d_mr = torch.full((R,), 30.0, dtype=torch.float64, device="cuda")
        for _ in range(2):
            g2.update_map_soa(d_start, d_dir, d_hit, d_mr, stream)
        torch.cuda.synchronize()
        ea.record(stream)
        g2.update_map_soa(d_start, d_dir, d_hit, d_mr, stream)
        eb.record(stream)
        torch.cuda.synchronize()
        ud_ms = ea.elapsed_time(eb)
        others["mapper update_map, device-resident scan (update_map_soa: two launches, no host sync)"] = {
            "value": R / (ud_ms * 1e-3), "unit": "rays/s", "total_ms": ud_ms}
        Q = 1 << 22
        qpos = torch.as_tensor(rngm.uniform(-25, 25, (3, Q)), dtype=torch.float64, device="cuda")
        qout = torch.empty(Q, dtype=torch.float64, device="cuda")
        gq = g2._grid()
        for _ in range(3):
            L.dart_map_query_batch(C.byref(gq), Q, Q, qpos.data_ptr(), qout.data_ptr(), stream.cuda_stream)
        ea.record(stream)
        L.dart_map_query_batch(C.byref(gq), Q, Q, qpos.data_ptr(), qout.data_ptr(), stream.cuda_stream)
        eb.record(stream)
        torch.cuda.synchronize()
        q_ms = ea.elapsed_time(eb)
        others["mapper query_occupancy: 4 Mi random queries on the 256^3 grid"] = {
            "value": Q / (q_ms * 1e-3), "unit": "queries/s", "kernel_ms": q_ms,
            "hbm_frac_streaming_part": (Q * 32) / (q_ms * 1e-3) / 1e9 / hbm_peak}
        line["other_configs"] = others
        # single-solve latency through the drop-in planner (metric's second half)
        planner = dp.SE3MPCPlanner.from_yaml()
        st = dp.DroneState(0.0, np.array([0.0, 0.0, 2.0]))
        planner.set_goal(np.array([10.0, 0.0, 5.0]))
        lat = []
        for i in range(260):
            t0 = time.perf_counter()
            planner.plan(st)
            lat.append((time.perf_counter() - t0) * 1e3)
        lat = lat[60:]
        line["single_solve_latency_ms"] = {"p50": statistics.median(lat), "p95": sorted(lat)[int(0.95 * len(lat))],
                                           "api": "SE3MPCPlanner.plan (host in, host out)", "n": len(lat)}
        # the same single problem on one host core through the CPU port (reported beside it: a GPU
        # does not win single-problem latency against a C port; the reference's own Python path
        # is 2.1 ms, BASELINE.md)
        p1 = np.array([[0.0, 0.0, 2.0]]); g1 = np.array([[10.0, 0.0, 5.0]])
        clat = []
        for i in range(260):
            t0 = time.perf_counter()
            oracle.solve_batch(oparams, p1, np.zeros((1, 3)), g1, nthreads=1)
            clat.append((time.perf_counter() - t0) * 1e3)
        line["single_solve_latency_ms"]["cpu_port_p50"] = statistics.median(clat[60:])
    sampler.stop()
    line["clocks"] = sampler.summary()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
