"""Reference tracking on the B200 (gradient_mode 7 = mode 3 with a per-timestep reference, 8 = mode 6
with it): every build that serves horizons <= 16 against the CPU restatement (tests/track_oracle)
under the rule of tests/test_gpu_kernel_matrix.py, with the exact checker; agreement with modes 3 / 6
when the reference is the goal at rest; the output paths; the closed loop along a path; the C ABI's
refusals on the device."""
import ctypes as C
import os

import numpy as np
import pytest

import track_exact
import track_oracle
from test_gpu_kernel_matrix import BUILDS, ROLLOUT_BUILDS, _hold_to_oracle, _kernel_info, _Sub, fingerprints  # noqa: F401
from test_gpu_spheres import _inputs, spheres_on_paths

pytestmark = pytest.mark.gpu

W, MARGIN = 1000.0, 0.5
CELLS = [(b, m) for b in ROLLOUT_BUILDS for m in (7, 8)]
ORACLE_SAMPLE, EXACT_SAMPLE = 2000, 24
# the goal at rest against modes 3 / 6: other kernels, which ptxas may contract differently
# (DESIGN.md 5e, test_gpu_spheres.test_unreachable_spheres_give_the_plain_bits)
REL_TOL = 1e-12


def _params(mode, N, tol=1e-3):
    import dart_planner_b200 as dp
    from dart_planner_b200.config import make_params
    return make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=tol, obstacle_weight=W),
                       gradient_mode=mode)


def reference(p0, N, seed, T=None):
    """A random walk of positions near the starts with random velocities, T = N + 3 samples; every
    eighth problem holds its start at rest (its solves stop on the projected gradient)."""
    rng = np.random.default_rng(seed)
    T = N + 3 if T is None else T
    P = p0[:, None] + rng.normal(0, 0.6, (len(p0), T, 3)).cumsum(1)
    V = rng.normal(0, 2, (len(p0), T, 3))
    P[::8], V[::8] = p0[::8, None], 0.0
    return P, V


def _solve(mode, N, p0, v0, hg, ref, start=0, spheres=None, x_warm=None, grid=None):
    from dart_planner_b200.planner import BatchWorkspace
    params = _params(mode, N)
    ws = BatchWorkspace(params, len(p0), pinned=False)
    ws.set_inputs_device(p0, v0, np.zeros_like(p0))
    ws.set_has_goal(hg)
    ws.set_warm(x_warm)
    ws.set_reference(ref[0], ref[1], start)
    if spheres is not None:
        ws.set_spheres((spheres[:, :3], spheres[:, 3]), MARGIN)
    if grid is not None:
        ws.set_map(grid, 0.2, 0.6)
    sol = ws.solve_device()
    return params, sol.numpy(), (None if grid is None else sol.first_hit.cpu().numpy())


def _oracle(oracle_mod, mode, N, p0, v0, hg, ref, start, spheres, x_warm=None):
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
    return track_oracle.solve_batch(op, mode, p0, v0, ref, start, spheres, W, MARGIN, has_goal=hg, x_warm=x_warm,
                                    nthreads=16)


def _explain(got, ref, alt):
    """Print the problems with equal counters that miss the tolerance, beside the oracle's own
    result after a one-ulp move of its inputs."""
    relf = np.abs(got.cost - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
    dx = np.abs(got.x - ref.x).max(axis=1)
    same = (got.nit == ref.nit) & (got.nfev == ref.nfev) & (got.status == ref.status)
    relf2 = np.abs(alt.cost - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
    dx2 = np.abs(alt.x - ref.x).max(axis=1)
    for i in np.where(same & ((dx > 1e-4) | (relf > 1e-5)))[0]:
        print(f"  problem {i}: dx {dx[i]:.3e} relf {relf[i]:.3e} cost {ref.cost[i]:.6e} nit {ref.nit[i]} "
              f"task {ref.task[i]}; oracle after one ulp: dx {dx2[i]:.3e} relf {relf2[i]:.3e} "
              f"nit {alt.nit[i]} nfev {alt.nfev[i]} (oracle nfev {ref.nfev[i]})")


@pytest.mark.parametrize("build,mode", CELLS, ids=[f"{BUILDS[b][0]}-mode{m}" for b, m in CELLS])
def test_track_cell_matches_the_oracle(oracle_mod, monkeypatch, fingerprints, build, mode):  # noqa: F811
    """At the build's largest horizon and at one that leaves lanes unused: cold, then warm from a
    tilted thrust history one sample further along the reference."""
    name, lanes, tpl, block, minb, Ns, B, variant = BUILDS[build]
    if variant is not None and "DART_SE3MPC_VARIANT" not in os.environ:
        monkeypatch.setenv("DART_SE3MPC_VARIANT", variant)
    rng = np.random.default_rng(build * 100 + mode)
    for N in (min(Ns[0], 16), Ns[1]):
        info = _kernel_info(_params(3, N), B)        # the build choice does not depend on the mode
        assert info == fingerprints[build], f"{name} N={N} B={B}: kernel_info {info}, the build's {fingerprints[build]}"
        p0, v0, _, hg = _inputs(B, 1000 * build + 10 * N + mode)
        v0[::8] = 0.0
        ref = reference(p0, N, build + N)
        s = spheres_on_paths(p0, v0, ref[0][:, -1]) if mode == 8 else None
        sub = np.arange(B) if B <= 3000 else np.unique(np.r_[np.arange(0, B, max(1, B // ORACLE_SAMPLE)), B - 1])
        xw, n_pg = None, {"cold": 0, "warm": 0}
        for start, st in ((0, "cold"), (1, "warm")):
            params, got, _ = _solve(mode, N, p0, v0, hg, ref, start, s, xw)
            refs = (ref[0][sub], ref[1][sub])
            r = _oracle(oracle_mod, mode, N, p0[sub], v0[sub], hg[sub], refs, start, s, None if xw is None else xw[sub])
            xws = None if xw is None else xw[sub]
            rerun = lambda: _oracle(oracle_mod, mode, N, np.nextafter(p0[sub], np.inf), v0[sub], hg[sub], refs,  # noqa
                                    start, s, None if xws is None else np.nextafter(xws, np.inf))
            what = f"{name} mode {mode} N {N} B {B} {st}"
            try:
                ok, same, escaped = _hold_to_oracle(3, st == "warm", _Sub(got, sub), r, rerun, what)
            except AssertionError:
                _explain(_Sub(got, sub), r, rerun())
                raise
            pick = np.r_[rng.choice(B, EXACT_SAMPLE, replace=False), np.where(got.task == 1)[0][:8]]
            n_pg[st] += track_exact.check_results(params, p0, v0, ref, start, hg, got, pick, s, W, MARGIN, what=what)
            print(f"{what}: ok {ok:.4f} same {same:.4f} {'one-ulp' if escaped else 'strict'}")
            if st == "cold":
                xw = got.x.copy()
                xw[:, 6 * N:] += rng.normal(0, 0.4, xw[:, 6 * N:].shape)      # tilted thrust history
                xw[::8] = got.x[::8]      # at rest on a reference that holds the start: stops at once
        assert n_pg["cold"] > 0 and n_pg["warm"] > 0, f"{name} mode {mode} N {N}: CONV_PGTOL stops checked {n_pg}"


@pytest.mark.parametrize("mode", [7, 8])
@pytest.mark.parametrize("build", [1, 5], ids=["latency", "throughput"])
def test_goal_reference_agrees_with_the_plain_modes(monkeypatch, build, mode):
    """r_k = goal, u_k = 0: the definition gives mode 3's (6's) bits; the kernels are other kernels,
    which ptxas may contract differently, so: identical counters, x and cost within REL_TOL."""
    from dart_planner_b200.planner import BatchWorkspace
    monkeypatch.delenv("DART_SE3MPC_VARIANT", raising=False)
    B, N = BUILDS[build][6], 8
    p0, v0, goal, hg = _inputs(B, 55 + mode)
    s = spheres_on_paths(p0, v0, goal) if mode == 8 else None
    ref = (np.repeat(goal[:, None], N, 1), None)
    xw = None
    for _ in range(2):
        ws = BatchWorkspace(_params(3 if mode == 7 else 6, N), B, pinned=False)
        ws.set_inputs_device(p0, v0, goal)
        ws.set_has_goal(hg)
        ws.set_warm(xw)
        if s is not None:
            ws.set_spheres((s[:, :3], s[:, 3]), MARGIN)
        plain = ws.solve_device().numpy()
        got = _solve(mode, N, p0, v0, hg, ref, 0, s, xw)[1]
        for a in ("nit", "nfev", "status", "task"):
            assert (getattr(got, a) == getattr(plain, a)).all(), a
        exact = np.mean([got.x[b].tobytes() == plain.x[b].tobytes() for b in range(B)])
        print(f"build {BUILDS[build][0]} mode {mode}: {exact:.4f} of the problems bit-identical")
        assert (np.abs(got.x - plain.x) <= REL_TOL * np.maximum(np.abs(plain.x), 1.0)).all()
        assert (np.abs(got.cost - plain.cost) <= REL_TOL * np.maximum(np.abs(plain.cost), 1.0)).all()
        xw = plain.x


@pytest.mark.parametrize("mode", [7, 8])
def test_output_paths_give_the_same_bits(oracle_mod, mode):
    """SoA output with and without the fused safety check; the throughput build (in-flight hint)
    agrees with the latency build as tests/test_gpu_rollout.py requires; plan_batch is the workspace."""
    import torch
    import dart_planner_b200 as dp
    from test_rollout_mode import _world
    N, B = 8, 3000
    p0, v0, _, hg = _inputs(B, 5)
    ref = reference(p0, N, 9, T=N)
    s = spheres_on_paths(p0, v0, ref[0][:, -1]) if mode == 8 else None
    og = _world(oracle_mod)
    grid = dp.DenseOccupancyGrid((128, 128, 128), (-64, -64, -64), 0.4)
    grid.occ.copy_(torch.from_numpy(og.occ))
    _, a, _ = _solve(mode, N, p0, v0, hg, ref, 0, s)
    _, b, hit = _solve(mode, N, p0, v0, hg, ref, 0, s, grid=grid)
    for f in ("x", "cost", "nit", "nfev", "status", "task", "accelerations", "attitudes", "body_rates", "thrusts"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f
    assert (hit >= -1).all() and (hit >= 0).any()
    with dp.planner.steps_in_flight(1 << 20):          # the throughput build
        thr = _solve(mode, N, p0, v0, hg, ref, 0, s)[1]
    assert (thr.nfev == a.nfev).mean() >= 0.999
    same = thr.nfev == a.nfev
    assert np.abs(thr.x - a.x)[same].max() <= 1e-9
    sph = None if s is None else (s[:, :3], s[:, 3])
    pb = dp.plan_batch(p0, v0, None, dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=1e-3,
                                                      obstacle_weight=W),
                       has_goal=hg, dynamics_consistent=True, reference=(torch.from_numpy(ref[0]).cuda(), ref[1]),
                       spheres=sph, sphere_margin=MARGIN, to_host=True)
    assert pb.x.tobytes() == a.x.tobytes() and pb.nfev.tobytes() == a.nfev.tobytes()


@pytest.mark.parametrize("mode", [7, 8])
def test_closed_loop_along_a_path(oracle_mod, mode):
    """Every step against the oracle from the same state with the window at the step index (the path
    has 10 samples: the last steps hold its end), sub-populations bit-identical to one run, and in
    mode 8 the collision record against the rasterised spheres."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from test_rollout_mode import _world
    from track_paths import circle_paths
    B, N, steps, T = 1024, 8, 14, 10
    P, V = circle_paths(B, T, 0.1)
    p0, v0 = P[:, 0].copy(), V[:, 0].copy()
    rng = np.random.default_rng(7)
    centers, radii = rng.uniform(-15, 15, (48, 3)), rng.uniform(0.8, 2.5, 48)
    s = np.c_[centers, radii] if mode == 8 else None
    params = _params(mode, N)
    og = _world(oracle_mod)
    cmap = dp.DenseOccupancyGrid((128, 128, 128), (-64, -64, -64), 0.4)
    cmap.occ.copy_(torch.from_numpy(og.occ))
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
    kw = dict(spheres=(centers, radii), sphere_margin=1.0) if mode == 8 else {}
    sims = []
    for parts in (1, 2):
        sim = ClosedLoopSim(params, B, plant_dt=0.1, reference_path=(P, V), collision_map=cmap, **kw)
        sim.reset(p0, v0)
        sims.append(sim)
    assert not sims[0].lateral_thrust_is_zero
    x = None

    class _Got:
        pass

    for k in range(steps):
        p, v = sims[0].positions().cpu().numpy().copy(), sims[0].velocities().cpu().numpy().copy()
        sims[0].step()
        r = track_oracle.solve_batch(op, mode, p, v, (P, V), k, s, W, 1.0, x_warm=x, nthreads=16)
        got = _Got()
        got.x, got.cost = sims[0].solution().cpu().numpy(), sims[0].cost[:B].cpu().numpy()
        got.nit, got.nfev, got.status = sims[0].meta[:, :B].cpu().numpy()
        xk = x
        rerun = lambda: track_oracle.solve_batch(op, mode, np.nextafter(p, np.inf), v, (P, V), k, s, W, 1.0,  # noqa
                                                 x_warm=None if xk is None else np.nextafter(xk, np.inf), nthreads=16)
        _hold_to_oracle(3, k > 0, got, r, rerun, f"closed loop mode {mode} step {k}")
        x = got.x
    sims[1].run(steps, parts=2)
    assert sims[0].state.cpu().numpy()[:, :B].tobytes() == sims[1].state.cpu().numpy()[:, :B].tobytes()
    assert sims[0].x.cpu().numpy()[:, :B].tobytes() == sims[1].x.cpu().numpy()[:, :B].tobytes()
    fc0, fc1 = sims[0].first_collision().cpu().numpy(), sims[1].first_collision().cpu().numpy()
    assert (fc0 == fc1).all() and ((fc0 >= -1) & (fc0 < steps)).all()


def test_refusals_on_the_device():
    """The refusals of the _track entries with real device buffers and a current device."""
    import torch
    from dart_planner_b200 import _cabi
    L = _cabi.lib()
    OK, BAD, UNS = _cabi.DART_OK, _cabi.DART_E_BADARG, _cabi.DART_E_UNSUPPORTED
    B, N = 64, 8
    buf = torch.zeros((64 * 9 * 4, B), dtype=torch.float64, device="cuda")
    bp = buf.data_ptr()
    lst = torch.zeros((2, 4), dtype=torch.float64, device="cuda")
    sph = _cabi.Spheres(2, 0, lst.data_ptr(), 0.5)
    ref = _cabi.TrackRef(N, 0, bp)

    def p(mode, n=N):
        q = _params(3, n)
        q.gradient_mode = mode
        return q

    def dev(q, r, s):
        return L.dart_se3mpc_solve_batch_track(C.byref(q), B, B, bp, bp, None, None, None, bp + 8 * 9 * N * B,
                                               *([None] * 9), None if r is None else C.byref(r),
                                               None if s is None else C.byref(s), None, 0.0, 0.0, None, None)

    def loop(q, r, s, warm=1, plant_dt=0.1):
        return L.dart_se3mpc_closed_loop_step_track(C.byref(q), B, B, bp, bp + 8 * 3 * B, None, bp + 8 * 6 * B, warm,
                                                    None, None, None, None, plant_dt, None if r is None else C.byref(r),
                                                    None if s is None else C.byref(s), None, 0.0, 0.6, 0, None, None)

    for call in (dev, loop):
        assert call(p(7), ref, None) == OK and call(p(8), ref, sph) == OK
        for mode in (0, 3, 5, 6, 9):
            assert call(p(mode), ref, None) == BAD and call(p(mode), ref, sph) == BAD
        assert call(p(7), None, None) == BAD and call(p(7), _cabi.TrackRef(N, 0, None), None) == BAD
        assert call(p(7), _cabi.TrackRef(0, 0, bp), None) == BAD and call(p(7), _cabi.TrackRef(N, -1, bp), None) == BAD
        assert call(p(7), ref, sph) == BAD and call(p(8), ref, None) == BAD
        assert call(p(7, 17), ref, None) == UNS and call(p(8, 17), ref, sph) == UNS
    assert loop(p(7), ref, None, warm=2) == BAD and loop(p(7), ref, None, plant_dt=0.05) == BAD
    torch.cuda.synchronize()
