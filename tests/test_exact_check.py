"""The exact-arithmetic checker (tests/exact_check.py) on the CPU oracles' results, in every gradient
mode, in a world whose horizons cross the grid's faces and corners; and a negative control that
proves check (a) has teeth.  The GPU tier (tests/test_gpu_kernel_matrix.py) runs the same checker
on the kernels' results."""
import numpy as np
import pytest

import exact_check as xc
import rollout_oracle
from edge_world import (EDGE_FREE, EDGE_ORIGIN, EDGE_PRIOR, EDGE_RES, EDGE_W, edge_box, edge_cells, edge_inputs,
                        exact_grid, oracle_grid, stationary_warm)


def _solve(oracle_mod, mode, N, p0, v0, goal, x_warm=None, og=None, free_level=EDGE_FREE):
    tol = 1e-3 if mode >= 3 else 5e-2
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=tol, consistent_gradient=int(mode == 1))
    kw = dict(grid=og, obstacle_weight=EDGE_W, free_level=free_level) if mode in (2, 4) else {}
    solve = rollout_oracle.solve_batch if mode >= 3 else oracle_mod.solve_batch
    return op, solve(op, p0, v0, goal, x_warm=x_warm, nthreads=8, **kw)


@pytest.mark.parametrize("mode,dtype", [(0, "float32"), (1, "float32"), (2, "float32"), (2, "float64"),
                                        (3, "float32"), (4, "float32"), (4, "float64")])
def test_checker_accepts_the_oracle(oracle_mod, mode, dtype):
    cells = edge_cells(dtype)
    og, eg = oracle_grid(oracle_mod, cells), exact_grid(cells)
    B = 96
    p0, v0, goal = edge_inputs(B, seed=10 + mode)
    hg = (np.arange(B) % 9 != 4).astype(np.uint8)
    pg = 0
    for N in (8, 5):
        op, cold = _solve(oracle_mod, mode, N, p0, v0, goal, og=og)
        xw = cold.x.copy()
        xw[:, 6 * N:] += np.random.default_rng(N).normal(0, 0.4, xw[:, 6 * N:].shape)
        xw = stationary_warm(xw, goal, N)
        _, warm = _solve(oracle_mod, mode, N, p0, v0, goal, x_warm=xw, og=og)
        for res, pin in ((cold, p0), (warm, p0)):
            pg += xc.check_results(op, mode, pin, v0, goal, None, res, range(0, B, 2), eg, EDGE_W, EDGE_FREE,
                                   what=f"oracle mode {mode} N {N}")
        if mode in (2, 4):
            # the horizons cross the grid: some positions read the prior, and the penalty is active
            lo, hi = edge_box()
            P = cold.x[:, :3 * N].reshape(B, N, 3)
            assert ((P < lo) | (P >= hi)).any(axis=2).any()
    assert pg > 0, "no CONV_PGTOL stop was checked"
    if mode != 2 and mode != 4:                 # problems without a goal
        op = oracle_mod.make_params(horizon=6, dt=0.1, consistent_gradient=int(mode == 1))
        solve = rollout_oracle.solve_batch if mode >= 3 else oracle_mod.solve_batch
        res = solve(op, p0, v0, goal, has_goal=hg, nthreads=8)
        xc.check_results(op, mode, p0, v0, goal, hg, res, range(B), what=f"has_goal mode {mode}")


@pytest.mark.parametrize("mode", [2, 4])
def test_checker_flags_a_shifted_grid_or_free_level(oracle_mod, mode):
    """Negative control: results computed with the grid's origin moved by one voxel, or with another
    free level, are checked against the unshifted definition.  Check (a) must flag them."""
    cells = edge_cells("float64")
    eg = exact_grid(cells)
    B, N = 96, 8
    p0, v0, goal = edge_inputs(B, seed=40 + mode)
    for og, fl in ((oracle_grid(oracle_mod, cells, (EDGE_ORIGIN[0] + 1,) + EDGE_ORIGIN[1:]), EDGE_FREE),
                   (oracle_grid(oracle_mod, cells), EDGE_FREE - 0.05)):
        op, res = _solve(oracle_mod, mode, N, p0, v0, goal, og=og, free_level=fl)
        err = np.array([xc.cost_error(op, mode, goal[b], res.x[b], res.cost[b], eg, EDGE_W, EDGE_FREE)
                        for b in range(B) if res.task[b] != xc.TASK_ABNORMAL])
        # problems whose horizons stay in free space cost the same under both definitions; the
        # others must be flagged
        assert (err > 1.0).sum() >= 8, f"only {(err > 1).sum()} of {err.size} flagged"
        # and the same results pass against the definition they were computed with
        ok = np.array([xc.cost_error(op, mode, goal[b], res.x[b], res.cost[b],
                                     xc.Grid(og.occ, (og.g.ox, og.g.oy, og.g.oz), EDGE_RES, EDGE_PRIOR), EDGE_W, fl)
                       for b in range(0, B, 3) if res.task[b] != xc.TASK_ABNORMAL])
        assert (ok <= 1.0).all()


def test_checker_flags_a_perturbed_rollout_and_a_false_stop(oracle_mod):
    """Checks (b) and (c) have teeth too: a P entry moved by 1e-12, and a CONV_PGTOL claim at a
    point whose projected gradient is large."""
    B, N = 16, 8
    p0, v0, goal = edge_inputs(B, seed=3)
    op, res = _solve(oracle_mod, 3, N, p0, v0, goal)
    x = res.x[0].copy()
    assert xc.rollout_ratio(op, p0[0], v0[0], x) <= 1.0
    x[3 * 5 + 1] += 1e-12
    assert xc.rollout_ratio(op, p0[0], v0[0], x) > 1.0
    x0 = oracle_mod.cold_start(op, p0[1], v0[1], goal[1])
    assert xc.projected_gradient_excess(op, 0, p0[1], v0[1], goal[1], x0) > op.gtol


def test_float64_cell_grids_refuse_the_mapper_queries(oracle_mod):
    """A grid of float64 cells serves the penalty only; the mapper queries read float32 cells and
    raise instead of reading through the empty float32 pointer."""
    og = oracle_grid(oracle_mod, edge_cells("float64"))
    for call in (lambda: og.query([0.0, 0.0, 0.0]), lambda: og.traj_safe(np.zeros((2, 3)), 1.0, 0.6),
                 lambda: og.add_sphere([0.0, 0.0, 0.0], 1.0)):
        with pytest.raises(TypeError):
            call()
    assert og.penalty([-5.0, 8.0, 3.0], EDGE_W, EDGE_FREE)[0] >= 0.0
    assert oracle_grid(oracle_mod, edge_cells("float32")).query([-5.0, 8.0, 3.0]).shape == (1,)
