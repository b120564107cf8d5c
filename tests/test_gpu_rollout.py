"""Dynamics-consistent solve mode on the GPU (gradient_mode 3 / 4): against the CPU oracle in every
lane configuration, properties of every output row, output paths, the grid-penalty variant and the
closed loop.  The mode is an extension (self-oracle: tests/rollout_oracle)."""
import ctypes as C

import numpy as np
import pytest

import rollout_oracle

from test_rollout_mode import GOAL_RADIUS, _configs4, _inputs, _plant_recursion_residual

pytestmark = pytest.mark.gpu


def _agree(got, ref, frac=0.99):
    same = (got.nit == ref.nit) & (got.nfev == ref.nfev) & (got.status == ref.status)
    assert same.mean() >= frac, f"counters agree on {same.mean():.4f}"
    dx = np.abs(got.x - ref.x).max(axis=1)
    relf = np.abs(got.cost - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
    # see tests/test_rollout_mode.py: a few long solves end in a flat valley (x to ~3e-4)
    assert (dx[same] <= 1e-4).mean() >= 0.995 and (relf[same] <= 1e-5).mean() >= 0.999
    return same


@pytest.mark.parametrize("N", [1, 4, 6, 8, 13, 16])
def test_matches_oracle_every_lane_configuration(oracle_mod, N):
    import dart_planner_b200 as dp
    B = 1000 + 7 * N                                   # ragged
    p0, v0, goal, hg = _inputs(B, seed=200 + N)
    tol = 1e-3
    cfg = dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=tol)
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=tol)
    xw = None
    for _ in range(2):                                 # cold, then warm at a shifted start
        ref = rollout_oracle.solve_batch(op, p0, v0, goal, has_goal=hg, x_warm=xw, nthreads=16)
        got = dp.plan_batch(p0, v0, goal, cfg, has_goal=hg, x_warm=xw, dynamics_consistent=True, to_host=True)
        _agree(got, ref)
        # properties of every row: a rollout from (p0, v0), thrusts in their box, cost = f(x)
        assert _plant_recursion_residual(got.x, p0, v0, N, 0.1) <= 1e-9
        T = got.x[:, 6 * N:].reshape(B, N, 3)
        assert (np.abs(T[..., :2]) <= op.tilt_thrust).all()
        assert ((T[..., 2] >= op.min_thrust) & (T[..., 2] <= op.max_thrust)).all()
        ok = got.task != 5
        fx = np.array([oracle_mod.objective(op, got.x[i], goal[i] if hg[i] else None) for i in range(B)])
        assert (np.abs(got.cost - fx)[ok] <= 1e-12 * np.abs(fx[ok])).all()
        xw = ref.x
        p0 = p0 + 0.1


def test_long_horizons_are_refused():
    """Horizons above 16 (32-lane groups) are not offered in these modes (DESIGN.md 5c)."""
    import dart_planner_b200 as dp
    p0, v0, goal, _ = _inputs(64)
    with pytest.raises(Exception):
        dp.plan_batch(p0, v0, goal, dp.SE3MPCConfig(prediction_horizon=20, dt=0.1), dynamics_consistent=True)


def test_output_paths_give_the_same_bits():
    """SoA, the packed rows and the host entry give the same bits; the throughput build (in-flight
    hint) agrees with the latency build to rounding (its register-capped code rounds differently)."""
    import dart_planner_b200 as dp
    from dart_planner_b200.config import make_params
    from dart_planner_b200.planner import BatchWorkspace, HostSolution
    N, B = 8, 3000
    p0, v0, goal, hg = _inputs(B, seed=5)
    pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=1e-3), gradient_mode=3)
    ws = BatchWorkspace(pr, B, pinned=True)
    ws.set_inputs_device(p0, v0, goal)
    ws.stage_host_inputs(p0, v0, goal)
    ref = ws.solve_device().numpy()
    got = HostSolution.from_packed_rows(N, ws.solve_rows().numpy())
    for f in ("x", "cost", "nit", "nfev", "status", "task", "accelerations", "attitudes", "body_rates", "thrusts"):
        np.testing.assert_array_equal(getattr(got, f), getattr(ref, f), err_msg=f)
    host = ws.solve_host(p0, v0, goal)
    np.testing.assert_array_equal(host.x, ref.x)
    with dp.planner.steps_in_flight(1 << 20):          # the throughput build
        thr = ws.solve_device().numpy()
    assert (thr.nfev == ref.nfev).mean() >= 0.999
    same = thr.nfev == ref.nfev
    assert np.abs(thr.x - ref.x)[same].max() <= 1e-9


def test_map_check_and_penalty_mode(oracle_mod):
    """Mode 4 (grid penalty on the rolled-out positions) against the oracle; the fused map check sees
    the rolled-out positions; the penalty does not raise the colliding fraction over mode 3."""
    import dart_planner_b200 as dp
    rng = np.random.default_rng(3)
    centers, radii = rng.uniform(-20, 20, (64, 3)), rng.uniform(0.5, 2.0, 64)
    grid = dp.DenseOccupancyGrid((128, 128, 128), (-64, -64, -64), 0.4)
    grid.add_obstacles(centers, radii)
    og = oracle_mod.DenseGrid((128, 128, 128), (-64, -64, -64), 0.4)
    for c, r in zip(centers, radii):
        og.add_sphere(c, r)
    B, N = 4096, 8
    p0, v0, goal, _ = _inputs(B, seed=8)
    cfg = dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=1e-3)
    m3 = dp.plan_batch(p0, v0, goal, cfg, grid=grid, safety_margin=1.0, collision_threshold=0.6,
                       dynamics_consistent=True).numpy()
    own = np.array([og.traj_safe(m3.positions[i], 1.0, 0.6) for i in range(B)])
    np.testing.assert_array_equal(m3.first_hit, own)
    m4 = dp.plan_batch(p0, v0, goal, cfg, grid=grid, safety_margin=1.0, collision_threshold=0.6,
                       dynamics_consistent=True, obstacle_penalty=True).numpy()
    ref = rollout_oracle.solve_batch(oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3),
                                 p0, v0, goal, nthreads=16, grid=og, obstacle_weight=cfg.obstacle_weight,
                                 free_level=0.5)
    _agree(m4, ref)
    assert (m4.first_hit >= 0).mean() <= (m3.first_hit >= 0).mean()
    with pytest.raises(ValueError):
        dp.plan_batch(p0[:4], v0[:4], goal[:4], cfg, dynamics_consistent=True, obstacle_penalty=True)


def test_closed_loop_step_against_the_cpu_loop(oracle_mod):
    """Every step against the oracle from the GPU's own state; with plant_dt == dt the state after a
    step is the plan's P_1 / V_1; sub-populations give the same bits as one launch per step."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    N, dt, B = 8, 0.1, 2048
    p0, v0, goal = _configs4(B)
    goal[:256] = p0[:256] + 0.02
    pr = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3), gradient_mode=3)
    op = oracle_mod.make_params(horizon=N, dt=dt, convergence_tolerance=1e-3)
    sim = ClosedLoopSim(pr, B, plant_dt=dt)
    sim.reset(p0, v0, goal)
    for s in range(15):
        pg, vg = sim.positions().cpu().numpy().copy(), sim.velocities().cpu().numpy().copy()
        xg = sim.solution().cpu().numpy().copy() if s > 0 else None
        sim.step()
        ref = rollout_oracle.solve_batch(op, pg, vg, goal, x_warm=xg, nthreads=16)
        meta = sim.meta[:, :B].cpu().numpy()
        got = type("R", (), dict(nit=meta[0], nfev=meta[1], status=meta[2], x=sim.solution().cpu().numpy(),
                                 cost=sim.cost[:B].cpu().numpy()))
        _agree(got, ref)
        np.testing.assert_allclose(sim.positions().cpu().numpy(), got.x[:, 3:6], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(sim.velocities().cpu().numpy(), got.x[:, 3 * N + 3:3 * N + 6], rtol=1e-12, atol=1e-14)
    # sub-populations in flight: same bits as one launch per step
    a = ClosedLoopSim(pr, B, plant_dt=dt)
    b = ClosedLoopSim(pr, B, plant_dt=dt)
    for s in (a, b):
        s.reset(p0, v0, goal)
    a.run(6, parts=1)
    b.run(6, parts=3)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(a.positions().cpu().numpy(), b.positions().cpu().numpy())
    np.testing.assert_array_equal(a.solution().cpu().numpy(), b.solution().cpu().numpy())
    # warm == 2 (no-tilt promise) is refused in mode 3; mode 4 has no map here
    L = _cabi.lib()
    st = sim.state
    rc = L.dart_se3mpc_closed_loop_step(C.byref(pr), B, sim.ld, st.data_ptr(), st.data_ptr() + 3 * 8 * sim.ld,
                                        st.data_ptr() + 6 * 8 * sim.ld, None, sim.x.data_ptr(), 2, None, None,
                                        None, None, dt, torch.cuda.current_stream().cuda_stream)
    assert rc == _cabi.DART_E_BADARG
    with pytest.raises(ValueError):
        ClosedLoopSim(make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt), gradient_mode=4), 16)


def test_closed_loop_reaches_goals():
    """configs[4] start distribution, 4 096 drones, 100 replans at tolerance 1e-3: every drone ends
    within the radius the CPU oracle's loop gives (tests/test_rollout_mode.py)."""
    import torch
    import dart_planner_b200 as dp
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    B, N, dt = 4096, 8, 0.1
    p0, v0, goal = _configs4(B)
    sim = ClosedLoopSim(make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=1e-3),
                                    gradient_mode=3), B, plant_dt=dt)
    sim.reset(p0, v0, goal)
    sim.run(100)
    torch.cuda.synchronize()
    d = np.linalg.norm(sim.positions().cpu().numpy() - goal, axis=1)
    assert d.max() <= GOAL_RADIUS, d.max()
