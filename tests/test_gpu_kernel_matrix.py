"""Every solve kernel the launcher can reach, against the CPU oracles, and the exact-arithmetic
checker (tests/exact_check.py) on its results.

`make_kernel_set` builds eight solve kernels per build: gradient modes 0, 1 and 2 with and without
tilt (the 9-slot kernel that serves warm starts, the 7-slot kernel that serves cold starts) and
modes 3 and 4 with tilt only.  Eleven builds give 88 kernels.  One cell here is one (build,
gradient mode) at two horizons -- the build's largest and one that leaves lanes or timestep slots
unused -- cold and then warm from a tilted thrust history, so each cell runs the 7- and the 9-slot
kernel of modes 0-2 and the only kernel of modes 3/4: 82 kernels in all.

Not covered: modes 3 and 4 on the 32-lane builds 3 (l32), 4 (l32x2) and 8 (l32_occ3).  The
library refuses these modes above horizon 16 (DESIGN.md 5c), so those six kernels are reachable
only through DART_SE3MPC_VARIANT at horizons a 16-lane build serves.

A cell takes the build's natural route where one exists (batch size and horizon; 6001 problems
for l8_occ3, 12288 + 5 for l16_occ3 / l32_occ3) and DART_SE3MPC_VARIANT otherwise, and asserts
the build that ran: `dart_se3mpc_kernel_info` with the same parameters, batch size and environment
must report that build's (lanes, block threads, shared memory, registers), which are checked to
tell all eleven builds apart.  The launcher ignores a variant too narrow for the horizon, and a
cell that fell back to the default build would be no coverage.  A DART_SE3MPC_VARIANT set in the
environment is left in force, so that, for example, `DART_SE3MPC_VARIANT=0 pytest -k l8_b64-mode0`
(l4 cannot hold N = 8: the launcher runs l8) fails on the build check.

Thresholds are those of the existing suite per mode: `_compare` of test_gpu_parity.py (modes
0/1; all counters cold, 99.5 % warm, 98 % in mode 1), the mode-2 rule of test_gpu_config3.py and
`_agree` of test_gpu_rollout.py (modes 3/4).  A run below them passes only where the configuration
is chaotic: the oracle itself misses the rule against its own result after a one-ulp move of its
inputs, and the kernel agrees with the oracle as well as the oracle agrees with itself
(test_gpu_parity_sweep.py); the rule's condition on problems with equal counters holds throughout.

The exact checker runs on a sample of every run, and check (c) must have met at least one
CONV_PGTOL stop of a cold and of a warm start per cell.  `-s` prints the table of the runs: the
fractions within tolerance and with equal counters, which rule held, and the stops checked."""
import ctypes as C
import os

import numpy as np
import pytest

import exact_check as xc
import rollout_oracle
from conftest import COST_RTOL, CTRL_ATOL
from edge_world import (EDGE_FREE, EDGE_ORIGIN, EDGE_PRIOR, EDGE_RES, EDGE_SHAPE, EDGE_W, edge_cells,
                        edge_inputs, exact_grid, oracle_grid, stationary_warm)

pytestmark = pytest.mark.gpu

# index: (name, lanes, timesteps per lane, block threads, resident blocks, horizons, B, variant)
BUILDS = {
    0: ("l4", 4, 1, 64, 2, (4, 3), 1001, None),
    1: ("l8", 8, 1, 128, 2, (8, 5), 1001, None),
    2: ("l16", 16, 1, 128, 2, (16, 9), 1001, None),
    3: ("l32", 32, 1, 128, 2, (32, 17), 1001, None),
    4: ("l32x2", 32, 2, 128, 2, (64, 33), 257, None),
    5: ("l8_occ3", 8, 1, 128, 3, (8, 5), 6001, None),
    6: ("l8_b64", 8, 1, 64, 6, (8, 5), 1001, "6"),
    7: ("l16_occ3", 16, 1, 128, 3, (16, 9), 12288 + 5, None),
    8: ("l32_occ3", 32, 1, 128, 3, (32, 17), 12288 + 5, None),
    9: ("l6", 6, 1, 128, 2, (6, 5), 1001, "9"),
    10: ("l6_occ5", 6, 1, 64, 5, (6, 5), 1001, "10"),
}
ROLLOUT_BUILDS = (0, 1, 2, 5, 6, 7, 9, 10)
CELLS = [(b, m) for b in BUILDS for m in (0, 1, 2)] + [(b, m) for b in ROLLOUT_BUILDS for m in (3, 4)]
ORACLE_SAMPLE = 2000          # problems of a large batch compared with the oracle
EXACT_SAMPLE = 24             # problems per solve run through the exact checker
_RAN = []


def _problems_per_block(lanes, block):
    return block // 32 * 5 if lanes == 6 else block // lanes     # 6-lane groups: five per warp


def _kernel_info(params, B):
    from dart_planner_b200 import _cabi
    info = [C.c_int32() for _ in range(5)]
    rc = _cabi.lib().dart_se3mpc_kernel_info(C.byref(params), B, *[C.byref(i) for i in info])
    assert rc == 0
    lanes, block, _, smem, regs = (i.value for i in info)
    return lanes, block, smem, regs


def _params(mode, N, tol=None, min_thrust=2.0):
    import dart_planner_b200 as dp
    from dart_planner_b200.config import make_params
    tol = tol if tol is not None else (1e-3 if mode >= 3 else 5e-2)
    cfg = dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, convergence_tolerance=tol, obstacle_weight=EDGE_W,
                          min_thrust=min_thrust)
    return make_params(cfg, gradient_mode=mode, obstacle_free_level=EDGE_FREE)


@pytest.fixture(scope="module")
def fingerprints():
    """(lanes, block, smem, regs) of every build, each reached by its own route; all distinct."""
    env = os.environ.pop("DART_SE3MPC_VARIANT", None)
    fp = {}
    try:
        for b, (_, lanes, tpl, block, minb, Ns, B, variant) in BUILDS.items():
            if variant is not None:
                os.environ["DART_SE3MPC_VARIANT"] = variant
            fp[b] = _kernel_info(_params(0, Ns[0]), B)
            os.environ.pop("DART_SE3MPC_VARIANT", None)
            got_lanes, got_block, smem, regs = fp[b]
            assert (got_lanes, got_block) == (lanes, block), BUILDS[b]
            ppb = _problems_per_block(lanes, block)
            assert smem % (8 * ppb) == 0 and smem // ppb == fp[0][2] // _problems_per_block(4, 64), BUILDS[b]
            # the launch bounds: minb resident blocks of `block` threads fit the register file
            assert 0 < regs <= 65536 // (minb * block) // 8 * 8, (BUILDS[b], regs)
            if minb == 3:
                assert regs <= 168, (BUILDS[b], regs)
    finally:
        if env is not None:
            os.environ["DART_SE3MPC_VARIANT"] = env
    assert len(set(fp.values())) == len(fp), f"two builds share a fingerprint: {fp}"
    return fp


@pytest.fixture(scope="module")
def coverage():
    yield _RAN
    lines = ["", f"{'build':<12}{'mode':>5}  {'start':<10}{'kernel':<8}{'N':>4}{'B':>7}  {'grid':<9}"
                 f"{'ok':>7}{'same':>7}  {'rule':<9}{'pgtol':>6}  kernel_info (lanes, block, smem, regs)"]
    for r in sorted(_RAN):
        lines.append(f"{r[1]:<12}{r[2]:>5}  {r[3]:<10}{r[4]:<8}{r[5]:>4}{r[6]:>7}  {r[7]:<9}"
                     f"{r[9]:>7.4f}{r[10]:>7.4f}  {'one-ulp' if r[11] else 'strict':<9}{r[12]:>6}  {r[8]}")
    kernels = {(r[0], r[2], r[4]) for r in _RAN}
    lines.append(f"{len(_RAN)} runs, {len(kernels)} distinct solve kernels, "
                 f"{sum(r[11] for r in _RAN)} runs under the one-ulp rule")
    print("\n".join(lines))


def _solve_gpu(mode, N, p0, v0, goal, hg, x_warm=None, grid=None, tol=None, min_thrust=2.0):
    from dart_planner_b200.planner import BatchWorkspace
    params = _params(mode, N, tol, min_thrust)
    ws = BatchWorkspace(params, len(p0), pinned=False)
    ws.set_inputs_device(p0, v0, goal)
    ws.set_has_goal(hg)
    ws.set_warm(x_warm)
    if mode in (2, 4):
        ws.set_map(None, penalty_grid=grid)
    return params, ws.solve_device().numpy()


def gpu_grid(cells):
    import torch
    import dart_planner_b200 as dp
    g = dp.DenseOccupancyGrid(EDGE_SHAPE, EDGE_ORIGIN, EDGE_RES, prior=EDGE_PRIOR,
                              dtype="float64" if cells.dtype == np.float64 else "float32")
    g.occ.copy_(torch.from_numpy(cells))
    return g


def _oracle(oracle_mod, mode, N, p0, v0, goal, hg, x_warm=None, og=None, tol=None, min_thrust=2.0):
    tol = tol if tol is not None else (1e-3 if mode >= 3 else 5e-2)
    op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=tol, consistent_gradient=int(mode == 1),
                                min_thrust=min_thrust)
    kw = dict(grid=og, obstacle_weight=EDGE_W, free_level=EDGE_FREE) if mode in (2, 4) else {}
    solve = rollout_oracle.solve_batch if mode >= 3 else oracle_mod.solve_batch
    return solve(op, p0, v0, goal, has_goal=hg, x_warm=x_warm, nthreads=16, **kw)


class _Sub:
    def __init__(self, r, idx):
        for k in ("x", "cost", "nit", "nfev", "status", "task", "attitudes", "thrusts", "accelerations"):
            setattr(self, k, np.asarray(getattr(r, k))[idx])


def _agreement(mode, warm, got, ref):
    """(passes, fraction ok, fraction with equal counters, same_ok) under the suite's rule for the
    mode; same_ok is the rule's condition on the problems with equal counters."""
    relf = np.abs(got.cost - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
    dx = np.abs(got.x - ref.x).max(axis=1)
    same = (got.nit == ref.nit) & (got.nfev == ref.nfev) & (got.status == ref.status)
    if mode >= 3:           # _agree, test_gpu_rollout.py
        ok = (dx <= 1e-4) & (relf <= 1e-5)
        same_ok = (dx[same] <= 1e-4).mean() >= 0.995 and (relf[same] <= 1e-5).mean() >= 0.999
        return same.mean() >= 0.99 and same_ok, ok.mean(), same.mean(), same_ok
    ok = (relf <= COST_RTOL) & (dx <= CTRL_ATOL)
    if mode == 2:           # test_grid_penalty_mode_matches_self_oracle, test_gpu_config3.py
        same_ok = bool(ok[same].all())
        return same.mean() >= 0.995 and same_ok, ok.mean(), same.mean(), same_ok
    frac = 0.98 if mode == 1 else (0.995 if warm else 1.0)      # _compare, test_gpu_parity.py
    same_ok = bool(ok[same].all()
                   and np.allclose(got.attitudes[same], ref.attitudes[same], rtol=0, atol=1e-6)
                   and np.allclose(got.thrusts[same], ref.thrusts[same], rtol=0, atol=1e-4)
                   and np.allclose(got.accelerations[same], ref.accelerations[same], rtol=0, atol=1e-4))
    return same.mean() >= frac and ok.mean() >= frac and same_ok, ok.mean(), same.mean(), same_ok


def _hold_to_oracle(mode, warm, got, ref, rerun, what):
    """The mode's rule; or, only where the configuration is chaotic -- the oracle itself misses the
    rule against its own result after a one-ulp move of its inputs -- agreement as good as the
    oracle's with itself (test_gpu_parity_sweep.py), with the rule's condition on the problems with
    equal counters kept.  Returns (fraction ok, fraction same, whether the one-ulp rule was used)."""
    passes, ok, same, same_ok = _agreement(mode, warm, got, ref)
    if passes:
        return ok, same, False
    assert same_ok, f"{what}: out of tolerance with equal counters (ok {ok:.4f} same {same:.4f})"
    alt = rerun()
    alt_passes, ok2, same2, _ = _agreement(mode, warm, alt, ref)
    assert not alt_passes, (f"{what}: misses the mode's rule (ok {ok:.4f} same {same:.4f}) where the oracle meets "
                            f"it against itself after one ulp (ok {ok2:.4f} same {same2:.4f})")
    slack = 2.0 / np.sqrt(len(ref.cost))
    assert ok >= ok2 - 0.03 - slack and same >= same2 - 0.06 - slack, \
        f"{what}: ok {ok:.4f} same {same:.4f}; the oracle against itself after one ulp: ok {ok2:.4f} same {same2:.4f}"
    return ok, same, True


def free_space_goals(eg, B, rng):
    """B positions inside the grid, off the voxel-centre planes, where the penalty is zero."""
    lo, hi = (np.array(EDGE_ORIGIN) * EDGE_RES, (np.array(EDGE_ORIGIN) + EDGE_SHAPE) * EDGE_RES)
    out = []
    while len(out) < B:
        q = rng.uniform(lo + 0.5, hi - 0.5)
        if xc.penalty(eg, EDGE_W, EDGE_FREE, q)[0] == 0 and xc.penalty(eg, EDGE_W, EDGE_FREE - 0.05, q)[0] == 0:
            out.append(q)
    return np.array(out)


def _run_cell(oracle_mod, monkeypatch, fingerprints, build, mode, N, B, variant, cells_dtype="float32",
              seed=0, tol=None):
    """Cold, then warm from the cold solution with tilted thrusts; returns the run rows."""
    name = BUILDS[build][0]
    if variant is not None and "DART_SE3MPC_VARIANT" not in os.environ:
        monkeypatch.setenv("DART_SE3MPC_VARIANT", variant)
    info = _kernel_info(_params(mode, N, tol), B)
    assert info == fingerprints[build], f"{name} N={N} B={B}: kernel_info {info}, the build's {fingerprints[build]}"
    cells = edge_cells(cells_dtype) if mode in (2, 4) else None
    grid, og, eg = (gpu_grid(cells), oracle_grid(oracle_mod, cells), exact_grid(cells)) if cells is not None \
        else (None, None, None)
    # starts at the goal stop on the projected gradient in modes 1, 3 and 4; in modes 0 and 2 they
    # end in the degenerate line-search regime, and the stationary warm starts take their place.
    # The cold 7-slot kernel of modes 0 and 2 gets its stops from a third run ("cold-stop"): every
    # problem at rest at its goal with min_thrust = m g, so that the cold start's hover thrust sits
    # on its bound and the reference gradient's projection vanishes there (in mode 2, with the
    # goal in free space).
    seed = 1000 * build + 10 * mode + N + seed
    p0, v0, goal = edge_inputs(B, seed=seed, at_goal=mode in (1, 3, 4))
    hg = (np.arange(B) % 11 != 3).astype(np.uint8)
    sub = np.arange(B) if B <= 3000 else np.unique(np.r_[np.arange(0, B, max(1, B // ORACLE_SAMPLE)), B - 1])
    rng = np.random.default_rng(build * 100 + mode * 10 + N)
    rows = []
    xw = None
    starts = ("cold", "warm", "cold-stop") if mode in (0, 2) else ("cold", "warm")
    for start in starts:
        min_thrust = 1.5 * 9.81 if start == "cold-stop" else 2.0
        if start == "warm" and mode in (0, 2):
            # the stationary warm starts are stationary only where the start is the goal at rest
            p0, v0 = p0.copy(), v0.copy()
            p0[::8], v0[::8] = goal[::8], 0.0
        if start == "cold-stop":
            if mode == 2:
                # goals in free space, where the penalty and its gradient vanish.  A start on the
                # penalty's kinks (voxel-centre planes, the levels where o crosses free_level) is
                # chaotic: the oracle's own result there moves beyond tolerance, with the same
                # counters, after a one-ulp move of the start.  The cold and warm runs above cover
                # the penalty's active region and the voxel-centre planes.
                goal = free_space_goals(eg, B, rng)
            p0, v0, xw = goal.copy(), np.zeros_like(v0), None
        params, got = _solve_gpu(mode, N, p0, v0, goal, hg, xw, grid, tol, min_thrust)
        kw = dict(og=og, tol=tol, min_thrust=min_thrust)
        ref = _oracle(oracle_mod, mode, N, p0[sub], v0[sub], goal[sub], hg[sub],
                      None if xw is None else xw[sub], **kw)
        xws = None if xw is None else xw[sub]
        rerun = lambda: _oracle(oracle_mod, mode, N, np.nextafter(p0[sub], np.inf), v0[sub], goal[sub],  # noqa: E731
                                hg[sub], None if xws is None else np.nextafter(xws, np.inf), **kw)
        what = f"{name} mode {mode} N {N} B {B} {start}"
        ok, same, escaped = _hold_to_oracle(mode, start == "warm", _Sub(got, sub), ref, rerun, what)
        pick = np.r_[rng.choice(B, EXACT_SAMPLE, replace=False), np.where(got.task == xc.TASK_PGTOL)[0][:8]]
        n_pg = xc.check_results(params, mode, p0, v0, goal, hg, got, pick, eg, EDGE_W, EDGE_FREE, what=what)
        kernel = "9-slot" if (start == "warm" or mode >= 3) else "7-slot"
        rows.append((build, name, mode, start, kernel, N, B, cells_dtype if cells is not None else "-", info,
                     ok, same, escaped, n_pg))
        if start == "cold":
            xw = got.x.copy()
            xw[:, 6 * N:] += rng.normal(0, 0.4, xw[:, 6 * N:].shape)      # tilted thrust history
            xw = stationary_warm(xw, goal, N)
    return rows


def _assert_stops_checked(rows, what):
    """Check (c) ran on at least one CONV_PGTOL stop of each start kind (cold, warm)."""
    for kind in ("cold", "warm"):
        n = sum(r[12] for r in rows if r[3].startswith(kind))
        assert n > 0, f"{what}: no CONV_PGTOL stop of a {kind} start was checked"


@pytest.mark.parametrize("build,mode", CELLS, ids=[f"{BUILDS[b][0]}-mode{m}" for b, m in CELLS])
def test_kernel_cell_matches_the_oracle(oracle_mod, monkeypatch, fingerprints, coverage, build, mode):
    name, lanes, tpl, block, minb, Ns, B, variant = BUILDS[build]
    rows = []
    for N in Ns:
        assert lanes * tpl >= N
        rows += _run_cell(oracle_mod, monkeypatch, fingerprints, build, mode, N, B, variant)
    coverage.extend(rows)
    _assert_stops_checked(rows, f"{name} mode {mode}")


def test_a_variant_too_narrow_for_the_horizon_is_detected(fingerprints, monkeypatch):
    """The launcher ignores DART_SE3MPC_VARIANT when the build cannot hold the horizon; the cells
    above would then see another build's fingerprint.  l4 asked for N = 8 runs l8."""
    monkeypatch.setenv("DART_SE3MPC_VARIANT", "0")
    assert _kernel_info(_params(0, 8), 1001) == fingerprints[1] != fingerprints[0]


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("build", [1, 5], ids=["latency", "throughput"])
@pytest.mark.parametrize("mode", [2, 4])
def test_grid_penalty_at_the_grid_edges(oracle_mod, monkeypatch, fingerprints, coverage, mode, build, dtype):
    """Modes 2 and 4 where horizons cross the faces and corners of a grid with an asymmetric origin,
    a prior above the free level (leaving the grid costs) and goal coordinates on voxel-centre
    planes; float32 and float64 cells; cold and warm; latency and throughput build."""
    B = BUILDS[build][6]
    rows = _run_cell(oracle_mod, monkeypatch, fingerprints, build, mode, 8, B, None, cells_dtype=dtype, seed=7)
    coverage.extend(rows)
    # one horizon only: stops are required over the test (the table shows them per run); the
    # matrix cells require them per start kind
    assert sum(r[12] for r in rows) > 0, f"grid edges mode {mode} {dtype}: no CONV_PGTOL stop was checked"


@pytest.mark.parametrize("mode", [1, 2, 3, 4])
def test_long_solves_first_changes_no_result_in_every_mode(oracle_mod, monkeypatch, fingerprints, mode):
    """The priority list ("long solves first") of cold batches of >= 16384 problems in a throughput
    build, in modes 1-4 (test_gpu_parity.py covers mode 0): identical bits with and without it
    (DART_SE3MPC_NO_PRIO), and the oracle's results on a sample."""
    monkeypatch.delenv("DART_SE3MPC_VARIANT", raising=False)
    B, N = 20000 + 3, 8
    assert _kernel_info(_params(mode, N), B) == fingerprints[5]           # l8_occ3: the list is built
    rng = np.random.default_rng(900 + mode)
    p0 = rng.uniform(-10, 10, (B, 3))
    v0 = rng.uniform(-1, 1, (B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], axis=1)
    near = rng.random(B) < 0.002
    near[:9000:1500] = True
    goal[near] = p0[near] + rng.normal(0, 0.25, (int(near.sum()), 3))
    hg = (np.arange(B) % 11 != 0).astype(np.uint8)
    cells = edge_cells("float32") if mode in (2, 4) else None
    grid = gpu_grid(cells) if cells is not None else None
    monkeypatch.delenv("DART_SE3MPC_NO_PRIO", raising=False)
    _, with_list = _solve_gpu(mode, N, p0, v0, goal, hg, grid=grid)
    monkeypatch.setenv("DART_SE3MPC_NO_PRIO", "1")
    _, without = _solve_gpu(mode, N, p0, v0, goal, hg, grid=grid)
    monkeypatch.delenv("DART_SE3MPC_NO_PRIO")
    for k in ("x", "cost", "nit", "nfev", "status", "task", "attitudes", "body_rates", "thrusts"):
        np.testing.assert_array_equal(getattr(with_list, k), getattr(without, k), err_msg=k)
    # the list is not empty: planted problems meet the launcher's near-goal predicate
    # (|goal - p0|^2 < w_thrust (m g)^2 N / w_pos, se3mpc_kernels.cu), in the first rounds and later
    r2 = 0.1 * (1.5 * 9.81) ** 2 * N / 100.0
    listed = ((goal - p0) ** 2).sum(axis=1) < r2
    assert listed[near & (hg != 0)].sum() >= 20 and listed[:9000].any() and listed[9000:].any()
    sub = np.r_[np.where(near)[0], rng.integers(0, B, 1500)]
    og = oracle_grid(oracle_mod, cells) if cells is not None else None
    kw = dict(og=og)
    ref = _oracle(oracle_mod, mode, N, p0[sub], v0[sub], goal[sub], hg[sub], **kw)
    rerun = lambda: _oracle(oracle_mod, mode, N, np.nextafter(p0[sub], np.inf), v0[sub], goal[sub], hg[sub], **kw)  # noqa: E731
    _hold_to_oracle(mode, False, _Sub(with_list, sub), ref, rerun, f"priority list mode {mode}")
