"""Signed distance, clearance field and the closed loop against a map on the GPU, against the
NumPy/SciPy restatements and the CPU oracles of tests/test_clearance_loop.py."""
import ctypes as C

import numpy as np
import pytest

import rollout_oracle

from test_clearance_loop import (ORIGIN, RES, SHAPE, clearance_field, field_grid, path_collides, signed_distance,
                                 signed_squared, sphere_world)
from test_gpu_closed_loop import _plant
from test_rollout_mode import GOAL_RADIUS

pytestmark = pytest.mark.gpu


def _device_grid(occ, origin=(0, 0, 0), res=0.3, prior=0.5):
    import torch
    import dart_planner_b200 as dp
    nz, ny, nx = occ.shape
    g = dp.DenseOccupancyGrid((nx, ny, nz), origin, res, prior=prior,
                              dtype="float64" if occ.dtype == np.float64 else "float32")
    g.occ.copy_(torch.from_numpy(np.ascontiguousarray(occ)))
    return g


def _random_grids():
    rng = np.random.default_rng(11)
    for shape in ((37, 20, 9), (1, 1, 50), (64, 3, 1), (33, 65, 17)):
        for frac in (0.02, 0.3, 0.8):
            occ = np.where(rng.random(shape) < frac, rng.uniform(0.61, 1.0, shape), rng.uniform(0.0, 0.6, shape))
            yield occ.astype(np.float32 if frac != 0.3 else np.float64)
    yield np.full((9, 10, 11), 0.5, np.float32)          # empty
    yield np.full((9, 10, 11), 0.9, np.float64)          # full
    t = np.full((12, 8, 5), 0.6, np.float32)             # exactly at the threshold: free
    t[3, 4, 2] = np.nextafter(np.float32(0.6), np.float32(1.0))
    yield t


def test_signed_distance_and_field_match_scipy():
    for occ in _random_grids():
        g = _device_grid(occ)
        phi = g.signed_distance(0.6).cpu().numpy()
        np.testing.assert_array_equal(g.squared_distance_voxels().cpu().numpy(), signed_squared(occ, 0.6))
        np.testing.assert_array_equal(phi, signed_distance(occ, 0.3, 0.6))
        f = g.clearance_field(0.7, 0.6)
        assert f.prob_prior == 0.5 and f.dtype == g.dtype and f.occ.shape == g.occ.shape
        np.testing.assert_array_equal(f.occ.cpu().numpy(), clearance_field(occ, 0.3, 0.6, 0.7))


def test_sphere_world_field(oracle_mod):
    """The 48-sphere world (128^3 at 0.4 m): the field the closed-loop tests fly against."""
    og = sphere_world(oracle_mod, B=1)[0]
    g = _device_grid(og.occ, ORIGIN, RES)
    np.testing.assert_array_equal(g.clearance_field(1.0).occ.cpu().numpy(), field_grid(oracle_mod, og, 1.0).occ)
    np.testing.assert_array_equal(g.squared_distance_voxels().cpu().numpy(), signed_squared(og.occ, 0.6))


def test_malformed_grids_are_refused():
    import torch
    from dart_planner_b200 import _cabi
    L = _cabi.lib()
    buf = torch.zeros(2 * 64, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    for bad in (_cabi.Grid(0, 4, 4, 0, 0, 0, 0.1, 0.5, buf.data_ptr(), 4, 0),
                _cabi.Grid(4, 4, 4, 0, 0, 0, 0.0, 0.5, buf.data_ptr(), 4, 0),
                _cabi.Grid(4, 4, 4, 0, 0, 0, 0.1, 0.5, None, 4, 0),
                _cabi.Grid(4, 4, 4, 0, 0, 0, 0.1, 0.5, buf.data_ptr(), 2, 0)):
        assert L.dart_map_signed_distance(C.byref(bad), 0.6, None, buf.data_ptr(), s) == _cabi.DART_E_BADARG
        assert L.dart_map_clearance_field(C.byref(bad), 0.6, 1.0, 0.5, buf.data_ptr(), buf.data_ptr(),
                                          s) == _cabi.DART_E_BADARG
    ok = _cabi.Grid(4, 4, 4, 0, 0, 0, 0.1, 0.5, buf.data_ptr(), 4, 0)
    assert L.dart_map_signed_distance(C.byref(ok), 0.6, None, None, s) == _cabi.DART_E_BADARG
    assert L.dart_map_clearance_field(C.byref(ok), 0.6, float("nan"), 0.5, buf.data_ptr(), buf.data_ptr(),
                                      s) == _cabi.DART_E_BADARG


def _world(oracle_mod, B):
    og, p0, goal = sphere_world(oracle_mod, B=B)
    occ = _device_grid(og.occ, ORIGIN, RES)
    return og, occ, occ.clearance_field(1.0), p0, goal


@pytest.mark.parametrize("mode", [4, 2])
def test_closed_loop_with_map_against_the_oracle(oracle_mod, mode):
    """Mode 4 on the clearance field and mode 2 on the occupancy itself: every step against the
    oracle from the GPU's own state; the plant step is exact; first_collision is the restated
    sampling of the GPU's own path history."""
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    N, dt, B, w = 8, 0.1, 1024, 1e5 if mode == 4 else 1e3
    og, occ, field, p0, goal = _world(oracle_mod, B)
    v0 = np.random.default_rng(5).uniform(-2, 2, (B, 3))
    pen_dev, pen_cpu = (field, field_grid(oracle_mod, og, 1.0)) if mode == 4 else (occ, og)
    tol = 1e-3 if mode == 4 else 5e-2
    pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=tol, obstacle_weight=w),
                     gradient_mode=mode)
    op = oracle_mod.make_params(horizon=N, dt=dt, convergence_tolerance=tol)
    margin = 1.0
    sim = ClosedLoopSim(pr, B, plant_dt=dt, penalty_grid=pen_dev, collision_map=occ, safety_margin=margin)
    sim.reset(p0, v0, goal)
    first = np.full(B, -1)
    solve = rollout_oracle.solve_batch if mode == 4 else oracle_mod.solve_batch
    for s in range(20):
        pg, vg = sim.positions().cpu().numpy().copy(), sim.velocities().cpu().numpy().copy()
        xg = sim.solution().cpu().numpy().copy() if s > 0 else None
        sim.step()
        ref = solve(op, pg, vg, goal, x_warm=xg, nthreads=16, grid=pen_cpu, obstacle_weight=w, free_level=0.5)
        meta = sim.meta[:, :B].cpu().numpy()
        xs = sim.solution().cpu().numpy()
        same = (meta[0] == ref.nit) & (meta[1] == ref.nfev) & (meta[2] == ref.status)
        assert same.mean() >= 0.99, f"step {s}: counters agree on {same.mean():.4f}"
        assert (np.abs(xs - ref.x).max(axis=1)[same] <= 1e-4).mean() >= 0.995, f"step {s}"
        p1, v1 = _plant(pg, vg, xs, N, dt)
        np.testing.assert_array_equal(sim.positions().cpu().numpy(), p1)
        np.testing.assert_array_equal(sim.velocities().cpu().numpy(), v1)
        hit = path_collides(og.occ, ORIGIN, RES, og.g.prior, pg, p1, margin, 0.6)
        first[hit & (first < 0)] = s
        np.testing.assert_array_equal(sim.first_collision().cpu().numpy(), first, err_msg=f"step {s}")
    if mode == 2:
        assert (first >= 0).any()      # the comparison saw collisions
    sim.reset(p0, v0, goal)
    assert (sim.first_collision().cpu().numpy() == -1).all()


def test_sub_populations_give_the_same_bits(oracle_mod):
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    N, dt, B = 8, 0.1, 8192
    og, occ, field, p0, goal = _world(oracle_mod, B)
    pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3, obstacle_weight=1e5),
                     gradient_mode=4)
    out = {}
    for parts in (1, None, 2, 3, 4):
        sim = ClosedLoopSim(pr, B, plant_dt=dt, penalty_grid=field, collision_map=occ, safety_margin=1.5)
        sim.reset(p0, np.zeros_like(p0), goal)
        sim.run(12, parts=parts)
        torch.cuda.synchronize()
        out[parts] = [t.cpu().numpy() for t in (sim.positions(), sim.solution(), sim.first_collision())]
    assert (out[1][2] >= 0).any()                     # a margin of 1.5 m: some paths come that close
    for parts in (None, 2, 3, 4):
        for a, b in zip(out[1], out[parts]):
            np.testing.assert_array_equal(a, b)


def test_clearance_field_flies_around_obstacles(oracle_mod):
    """4 096 drones, 100 replans: mode 3 collides for at least 5 % (CPU oracle, 256 drones: 9.4 %;
    measured here: 13.7 %).  Mode 4 on the 1 m clearance field (w 1e5) collided for none of the
    oracle's 256 drones, but for 1 of these 4 096 (DESIGN.md 5d): at most one in a thousand.  Every
    mode-3 drone and all but a few detouring mode-4 drones end within 1e-4 m of their goals (two of
    the 4 096 mode-4 drones were not, the farther 2.5e-3 m away after 100 replans)."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    N, dt, B = 8, 0.1, 4096
    og, occ, field, p0, goal = _world(oracle_mod, B)
    rate = {}
    for mode in (3, 4):
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3,
                                         obstacle_weight=1e5), gradient_mode=mode)
        sim = ClosedLoopSim(pr, B, plant_dt=dt, penalty_grid=field if mode == 4 else None, collision_map=occ)
        sim.reset(p0, np.zeros_like(p0), goal)
        sim.run(100)
        torch.cuda.synchronize()
        rate[mode] = (sim.first_collision().cpu().numpy() >= 0).mean()
        d = np.linalg.norm(sim.positions().cpu().numpy() - goal, axis=1)
        print(f"mode {mode}: collided {rate[mode]:.4f}, within {GOAL_RADIUS:g} m {(d <= GOAL_RADIUS).mean():.4f}, "
              f"max {d.max():.3g} m")
        if mode == 3:
            assert d.max() <= GOAL_RADIUS, d.max()
        else:
            assert (d <= GOAL_RADIUS).mean() >= 0.999 and d.max() <= 1e-2, d.max()
    assert rate[4] <= 1e-3 and rate[3] >= 0.05, rate


def test_refusals(oracle_mod):
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    L = _cabi.lib()
    B, N, dt = 64, 8, 0.1
    occ = _device_grid(np.full((8, 8, 8), 0.5, np.float32), (-4, -4, -4), 0.5)
    for mode in (2, 4):
        with pytest.raises(ValueError):
            ClosedLoopSim(make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt), gradient_mode=mode), B)
    sim = ClosedLoopSim(make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt), gradient_mode=3), B,
                        collision_map=occ)
    st, ld, s = sim.state, sim.ld, torch.cuda.current_stream().cuda_stream
    g = occ._grid()
    fc = sim._first_collision.data_ptr()

    def step_map(mode, warm, pen, chk, first):
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt), gradient_mode=mode)
        return L.dart_se3mpc_closed_loop_step_map(
            C.byref(pr), B, ld, st.data_ptr(), st.data_ptr() + 3 * 8 * ld, st.data_ptr() + 6 * 8 * ld, None,
            sim.x.data_ptr(), warm, None, None, None, None, dt, pen, chk, 0.0, 0.6, 0, first, s)

    def step_old(mode):
        pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt), gradient_mode=mode)
        return L.dart_se3mpc_closed_loop_step(
            C.byref(pr), B, ld, st.data_ptr(), st.data_ptr() + 3 * 8 * ld, st.data_ptr() + 6 * 8 * ld, None,
            sim.x.data_ptr(), 0, None, None, None, None, dt, s)

    for mode in (2, 4):
        assert step_map(mode, 0, None, None, None) == _cabi.DART_E_BADARG        # no penalty grid
        assert step_old(mode) == _cabi.DART_E_UNSUPPORTED                           # the old entry
    assert step_map(3, 2, None, None, None) == _cabi.DART_E_BADARG                  # warm == 2
    assert step_map(4, 2, C.byref(g), None, None) == _cabi.DART_E_BADARG
    assert step_map(3, 0, None, C.byref(g), None) == _cabi.DART_E_BADARG            # not together
    assert step_map(3, 0, None, None, fc) == _cabi.DART_E_BADARG
    bad = _cabi.Grid(8, 8, 8, -4, -4, -4, 0.5, 0.5, occ.occ.data_ptr(), 3, 0)
    assert step_map(3, 0, None, C.byref(bad), fc) == _cabi.DART_E_BADARG
    assert step_map(4, 0, C.byref(bad), None, None) == _cabi.DART_E_BADARG
    assert step_map(3, 0, None, C.byref(g), fc) == _cabi.DART_OK
    torch.cuda.synchronize()


def test_plan_batch_with_a_penalty_grid(oracle_mod):
    """The penalty reads penalty_grid (same bits as passing the field as the grid), and the safety
    check of `grid` (a second launch) gives what trajectories_safe_soa gives on the solved x."""
    import dart_planner_b200 as dp
    B, N = 4096, 8
    og, occ, field, p0, goal = _world(oracle_mod, B)
    v0 = np.random.default_rng(6).uniform(-2, 2, (B, 3))
    cfg = dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=1e-3, obstacle_weight=1e5)
    sol = dp.plan_batch(p0, v0, goal, cfg, grid=occ, penalty_grid=field, obstacle_penalty=True,
                        dynamics_consistent=True, safety_margin=0.5)
    own = occ.trajectories_safe_soa(sol.out[: 3 * N], B, N, 0.5, 0.6)[:B]
    np.testing.assert_array_equal(sol.first_hit.cpu().numpy(), own.cpu().numpy())
    same = dp.plan_batch(p0, v0, goal, cfg, grid=field, obstacle_penalty=True, dynamics_consistent=True).numpy()
    np.testing.assert_array_equal(sol.numpy().x, same.x)
    ref = rollout_oracle.solve_batch(oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3),
                                     p0, v0, goal, nthreads=16, grid=field_grid(oracle_mod, og, 1.0),
                                     obstacle_weight=1e5, free_level=0.5)
    agree = (same.nit == ref.nit) & (same.nfev == ref.nfev)
    assert agree.mean() >= 0.99
    with pytest.raises(ValueError):
        dp.plan_batch(p0[:4], v0[:4], goal[:4], cfg, penalty_grid=field)
