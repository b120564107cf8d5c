"""Sphere obstacle penalty on the B200 (gradient_mode 5 / 6): every solve build against the CPU
restatement (tests/sphere_oracle) under the rule of tests/test_gpu_kernel_matrix.py, the exact
checker, bit-equality with modes 0 / 3 where no sphere is reached, the host entry against the device
entry on its three staging paths, the drop-in planner with the mapper bridge's spheres, and the
closed loop."""
import os

import numpy as np
import pytest

import sphere_exact
import sphere_oracle
from test_gpu_kernel_matrix import BUILDS, ROLLOUT_BUILDS, _hold_to_oracle, _kernel_info, _Sub, fingerprints  # noqa: F401

pytestmark = pytest.mark.gpu

W, MARGIN = 1000.0, 0.5
CELLS = [(b, 5) for b in BUILDS] + [(b, 6) for b in ROLLOUT_BUILDS]
ORACLE_SAMPLE, EXACT_SAMPLE = 2000, 24
# unreachable spheres against the plain kernel: the same solve up to the rounding of the few
# operations ptxas contracts differently (see test_unreachable_spheres_give_the_plain_bits)
REL_TOL = 1e-12


def _params(mode, N, tol=None):
    import dart_planner_b200 as dp
    from dart_planner_b200.config import make_params
    tol = tol if tol is not None else (1e-3 if mode in (3, 6) else 5e-2)
    return make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=tol, obstacle_weight=W),
                       gradient_mode=mode)


def _inputs(B, seed):
    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-10, 10, (B, 3))
    v0 = rng.uniform(-2, 2, (B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], axis=1)
    p0[::8], v0[::8] = goal[::8], 0.0                      # at rest at the goal: projected-gradient stops
    hg = (np.arange(B) % 11 != 3).astype(np.uint8)
    return p0, v0, goal, hg


def spheres_on_paths(p0, v0, goal, n=20, seed=5):
    """n spheres where plans go: on start-goal segments (mode 5) and along the initial velocity (mode 6)."""
    rng = np.random.default_rng(seed)
    i = rng.choice(np.where(np.arange(len(p0)) % 8 != 0)[0], n, replace=False)
    c = np.where((np.arange(n) % 2 == 0)[:, None], 0.5 * (p0[i] + goal[i]), p0[i] + 0.4 * v0[i])
    return sphere_oracle.sphere_list(c + rng.normal(0, 0.2, (n, 3)), rng.uniform(0.6, 1.6, n))


def _solve(mode, N, p0, v0, goal, hg, spheres, x_warm=None, tol=None):
    from dart_planner_b200.planner import BatchWorkspace
    params = _params(mode, N, tol)
    ws = BatchWorkspace(params, len(p0), pinned=False)
    ws.set_inputs_device(p0, v0, goal)
    ws.set_has_goal(hg)
    ws.set_warm(x_warm)
    if spheres is not None:
        ws.set_spheres((spheres[:, :3], spheres[:, 3]), MARGIN)
    return params, ws.solve_device().numpy()


def _oracle(oracle_mod, mode, N, p0, v0, goal, hg, spheres, x_warm=None, tol=None):
    tol = tol if tol is not None else (1e-3 if mode == 6 else 5e-2)
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=tol)
    return sphere_oracle.solve_batch(op, mode, p0, v0, goal, spheres, W, MARGIN, has_goal=hg, x_warm=x_warm,
                                     nthreads=16)


@pytest.mark.parametrize("build,mode", CELLS, ids=[f"{BUILDS[b][0]}-mode{m}" for b, m in CELLS])
def test_sphere_cell_matches_the_oracle(oracle_mod, monkeypatch, fingerprints, build, mode):  # noqa: F811
    """Cold (mode 5: the 7-slot kernel) and warm (the 9-slot kernel, from a tilted thrust history in
    mode 6 and from the cold solution in mode 5) at the build's largest allowed horizon."""
    name, lanes, tpl, block, minb, Ns, B, variant = BUILDS[build]
    N = min(Ns[0], 16) if mode == 6 else Ns[0]
    if variant is not None and "DART_SE3MPC_VARIANT" not in os.environ:
        monkeypatch.setenv("DART_SE3MPC_VARIANT", variant)
    info = _kernel_info(_params(0, N), B)            # the build choice does not depend on the mode
    assert info == fingerprints[build], f"{name} N={N} B={B}: kernel_info {info}, the build's {fingerprints[build]}"
    p0, v0, goal, hg = _inputs(B, 1000 * build + mode)
    s = spheres_on_paths(p0, v0, goal)
    sub = np.arange(B) if B <= 3000 else np.unique(np.r_[np.arange(0, B, max(1, B // ORACLE_SAMPLE)), B - 1])
    rng = np.random.default_rng(build * 100 + mode)
    xw, n_pg, touched = None, 0, 0.0
    for start in ("cold", "warm"):
        params, got = _solve(mode, N, p0, v0, goal, hg, s, xw)
        ref = _oracle(oracle_mod, mode, N, p0[sub], v0[sub], goal[sub], hg[sub], s, None if xw is None else xw[sub])
        xws = None if xw is None else xw[sub]
        rerun = lambda: _oracle(oracle_mod, mode, N, np.nextafter(p0[sub], np.inf), v0[sub], goal[sub], hg[sub],  # noqa
                                s, None if xws is None else np.nextafter(xws, np.inf))
        what = f"{name} mode {mode} N {N} B {B} {start}"
        ok, same, escaped = _hold_to_oracle(2 if mode == 5 else 3, start == "warm", _Sub(got, sub), ref, rerun, what)
        pick = np.r_[rng.choice(B, EXACT_SAMPLE, replace=False), np.where(got.task == 1)[0][:8]]
        n_pg += sphere_exact.check_results(params, mode, p0, v0, goal, hg, got, pick, s, W, MARGIN, what=what)
        if mode == 5:
            assert (got.x[:, 6 * N:].reshape(B, N, 3)[..., :2] == 0).all() or start == "warm"
        print(f"{what}: ok {ok:.4f} same {same:.4f} {'one-ulp' if escaped else 'strict'}")
        if start == "cold":
            plain = _solve(0 if mode == 5 else 3, N, p0, v0, goal, hg, None)[1]
            touched = (np.abs(got.x - plain.x).max(axis=1) > 1e-6).mean()
            xw = got.x.copy()
            if mode == 6:
                xw[:, 6 * N:] += rng.normal(0, 0.4, xw[:, 6 * N:].shape)      # tilted thrust history
    assert touched >= 0.03, f"{name} mode {mode}: only {touched:.3f} of the plans meet a sphere"
    if mode == 6:
        assert n_pg > 0, f"{name} mode 6: no CONV_PGTOL stop was checked"


@pytest.mark.parametrize("mode", [5, 6])
@pytest.mark.parametrize("build", [1, 5], ids=["latency", "throughput"])
def test_unreachable_spheres_give_the_plain_bits(monkeypatch, build, mode):
    """An empty list runs mode 0's / 3's own kernel: every output bit for bit.  Unreachable spheres
    add +0 to f and -0 to the gradient, so the host build of the core returns exactly the plain bits
    (tests/test_sphere_mode.py); the mode-5 / 6 kernels, though, are other kernels, and ptxas contracts
    the plain (not DP_MUL / DP_ADD) products and sums of the shared solver code kernel by kernel: in
    the breakpoint walk's f1 = f1 + dt f2 + dibp^2 - theta dibp zibp, one unrolled copy fuses dibp^2
    into an FMA in the l8_occ3 mode-6 kernel and rounds it separately in mode 3 (SASS per source
    line).  Such a difference moves a result by roundings; on a B200 it changed no decision the
    counters record, and the test requires that: the counters must be identical on every problem, and x and cost within REL_TOL of the plain kernel's (relative to max(|v|, 1))."""
    monkeypatch.delenv("DART_SE3MPC_VARIANT", raising=False)
    B = BUILDS[build][6]
    p0, v0, goal, hg = _inputs(B, 77 + mode)
    far = sphere_oracle.sphere_list([[500.0, 500.0, 500.0], [-400.0, 0.0, 0.0]], [1.0, 2.0])
    xw = None
    for _ in range(2):
        plain = _solve(0 if mode == 5 else 3, 8, p0, v0, goal, hg, None, xw)[1]
        got = _solve(mode, 8, p0, v0, goal, hg, np.zeros((0, 4)), xw)[1]
        for a in ("x", "cost", "nit", "nfev", "status", "task", "attitudes", "body_rates", "thrusts"):
            assert getattr(got, a).tobytes() == getattr(plain, a).tobytes(), a
        got = _solve(mode, 8, p0, v0, goal, hg, far, xw)[1]
        for a in ("nit", "nfev", "status", "task"):
            assert (getattr(got, a) == getattr(plain, a)).all(), a
        exact = np.mean([got.x[b].tobytes() == plain.x[b].tobytes() for b in range(B)])
        print(f"build {BUILDS[build][0]} mode {mode}: {exact:.4f} of the problems bit-identical")
        assert (np.abs(got.x - plain.x) <= REL_TOL * np.maximum(np.abs(plain.x), 1.0)).all()
        assert (np.abs(got.cost - plain.cost) <= REL_TOL * np.maximum(np.abs(plain.cost), 1.0)).all()
        xw = plain.x


@pytest.mark.parametrize("B", [1, 600, 65541])
@pytest.mark.parametrize("mode", [5, 6])
def test_host_entry_equals_device_entry(B, mode):
    """The mapped pinned block (1), the staged workspace (600) and the chunked two-stream path
    (65 541): the sphere list reaches every chunk."""
    import ctypes as C
    from dart_planner_b200 import _cabi
    N = 8
    p0, v0, goal, hg = _inputs(B, 5 + B)
    s = spheres_on_paths(p0, v0, goal, n=min(20, B)) if B > 20 else sphere_oracle.sphere_list(
        [0.5 * (p0[0] + goal[0])], [1.5])
    params, dev = _solve(mode, N, p0, v0, goal, None, s)
    out = {k: np.zeros(sh) for k, sh in (("x", (9 * N, B)), ("cost", (1, B)), ("acc", (3 * N, B)), ("att", (3 * N, B)),
                                          ("rates", (3 * N, B)), ("thr", (N, B)))}
    meta = np.zeros((3, B), np.int32)
    soa = lambda a: np.ascontiguousarray(a.T)  # noqa: E731
    ins = [soa(p0), soa(v0), soa(goal)]
    sph = _cabi.Spheres(len(s), 0, s.ctypes.data, MARGIN)
    rc = _cabi.lib().dart_se3mpc_solve_batch_host_spheres(
        C.byref(params), B, *[a.ctypes.data for a in ins], None, None, out["x"].ctypes.data, out["cost"].ctypes.data,
        meta[0].ctypes.data, meta[1].ctypes.data, meta[2].ctypes.data, out["acc"].ctypes.data, out["att"].ctypes.data,
        out["rates"].ctypes.data, out["thr"].ctypes.data, C.byref(sph))
    _cabi.check(rc, "dart_se3mpc_solve_batch_host_spheres")
    assert out["x"].T.tobytes() == np.ascontiguousarray(dev.x).tobytes()
    assert out["cost"][0].tobytes() == np.ascontiguousarray(dev.cost).tobytes()
    assert (meta[0] == dev.nit).all() and (meta[1] == dev.nfev).all() and (meta[2] == dev.status).all()
    assert out["att"].T.reshape(B, N, 3).tobytes() == np.ascontiguousarray(dev.attitudes).tobytes()


def test_drop_in_planner_with_the_mapper_bridge(oracle_mod):
    """refresh_obstacles_from_mapper, then plan() with avoid_obstacles=True: the oracle's mode 5 on
    the same problem; avoid_obstacles=False: today's bits; update_plan with an obstacle on the plan
    changes the plan."""
    import dart_planner_b200 as dp
    from dart_planner_b200.planner import SE3MPCPlanner
    from dart_planner_b200.types import DroneState
    from conftest import load_golden
    from test_gpu_mapper import _bridge_map
    d = load_golden("local_grid")
    mapper, center, kw = _bridge_map(dp, d, "float64"), d["center"], dict(size=float(d["size"]))
    cfg = dp.SE3MPCConfig(prediction_horizon=8, dt=0.1, convergence_tolerance=1e-3)
    state = DroneState(timestamp=0.0, position=np.asarray(center, np.float64) + [-4.0, 0.3, 0.0],
                       velocity=np.array([1.0, 0.0, 0.0]))
    goal = np.asarray(center, np.float64) + [4.0, 0.3, 0.0]
    plans = {}
    for avoid in (False, True):
        pl = SE3MPCPlanner(cfg, respect_config_dt=True, avoid_obstacles=avoid)
        n = pl.refresh_obstacles_from_mapper(mapper, center, **kw)
        assert n > 0
        pl.set_goal(goal)
        plans[avoid] = pl.plan(state)
        if avoid:
            s = np.array([[*c, r] for c, r in pl.obstacles])
            op = oracle_mod.make_params(horizon=8, dt=0.1, convergence_tolerance=1e-3)
            ref = sphere_oracle.solve_batch(op, 5, state.position[None], state.velocity[None], goal[None], s,
                                            cfg.obstacle_weight, cfg.safety_margin)
            assert pl.last_result["nit"] == ref.nit[0] and pl.last_result["nfev"] == ref.nfev[0]
            np.testing.assert_allclose(pl.last_result["x"], ref.x[0], rtol=0, atol=1e-6)
    plain = SE3MPCPlanner(cfg, respect_config_dt=True)
    plain.set_goal(goal)
    today = plain.plan(state)
    for k in today:
        assert today[k].tobytes() == plans[False][k].tobytes(), k
    # update_plan with one obstacle on the straight plan moves the plan
    pl = SE3MPCPlanner(cfg, respect_config_dt=True, avoid_obstacles=True)
    pl.set_goal(goal)
    free = pl.plan(state)["positions"].copy()
    pl.update_plan(state, [{"position": free[4] + [0.0, 0.2, 0.0], "radius": 0.5}])
    moved = pl.last_result["x"][:24].reshape(8, 3)
    assert np.abs(moved - free).max() > 1e-3


@pytest.mark.parametrize("mode", [5, 6])
def test_closed_loop_with_spheres(oracle_mod, mode):
    """Every step against the oracle from the same state, sub-populations bit-identical to one run,
    and the collision record against the rasterised spheres."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from test_rollout_mode import _configs4, _world
    B, N, steps = 1024, 8, 12
    p0, v0, goal = _configs4(B)
    rng = np.random.default_rng(7)
    centers, radii = rng.uniform(-15, 15, (48, 3)), rng.uniform(0.8, 2.5, 48)
    s = sphere_oracle.sphere_list(centers, radii)
    params = _params(mode, N, tol=1e-3)
    og = _world(oracle_mod)
    cmap = dp.DenseOccupancyGrid((128, 128, 128), (-64, -64, -64), 0.4)
    cmap.occ.copy_(torch.from_numpy(og.occ))
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
    sims = []
    for parts in (1, 2):
        sim = ClosedLoopSim(params, B, plant_dt=0.1, spheres=(centers, radii), sphere_margin=1.0, collision_map=cmap)
        sim.reset(p0, v0, goal)
        sims.append(sim)
    assert sims[0].lateral_thrust_is_zero == (mode == 5)
    x = None

    class _Got:
        pass

    for k in range(steps):
        p, v = sims[0].positions().cpu().numpy().copy(), sims[0].velocities().cpu().numpy().copy()
        sims[0].step()
        ref = sphere_oracle.solve_batch(op, mode, p, v, goal, s, W, 1.0, x_warm=x, nthreads=16)
        got = _Got()
        got.x, got.cost = sims[0].solution().cpu().numpy(), sims[0].cost[:B].cpu().numpy()
        got.nit, got.nfev, got.status = sims[0].meta[:, :B].cpu().numpy()
        xk = x
        rerun = lambda: sphere_oracle.solve_batch(op, mode, np.nextafter(p, np.inf), v, goal, s, W, 1.0,  # noqa
                                                  x_warm=None if xk is None else np.nextafter(xk, np.inf), nthreads=16)
        # tolerance 1e-3: the closed-loop rule of tests/test_gpu_rollout.py in both modes (with spheres,
        # mode 5 also ends solves by the ftol rule in flat valleys, where x is determined to ~1e-3)
        _hold_to_oracle(3, k > 0, got, ref, rerun, f"closed loop mode {mode} step {k}")
        x = got.x
    sims[1].run(steps, parts=2)
    sims[1].run(0)
    assert sims[0].state.cpu().numpy()[:, :B].tobytes() == sims[1].state.cpu().numpy()[:, :B].tobytes()
    assert sims[0].x.cpu().numpy()[:, :B].tobytes() == sims[1].x.cpu().numpy()[:, :B].tobytes()
    fc0, fc1 = sims[0].first_collision().cpu().numpy(), sims[1].first_collision().cpu().numpy()
    assert (fc0 == fc1).all()
    assert ((fc0 >= -1) & (fc0 < steps)).all()
