"""SciPy's L-BFGS-B options away from their defaults in every solve build, against the CPU oracles
(tests/test_solver_options.py has the option sets and the CPU tier).

One cell is one (build, gradient mode, option set): every build in modes 0-2 and ROLLOUT_BUILDS in
modes 3/4, at the build's largest horizon (test_gpu_kernel_matrix.py covers partial horizons),
solved cold (the 7-slot kernel in modes 0-2) and then warm from a tilted thrust history (the 9-slot
kernel), at every setting `settings(mode)` lists.  Each run is held to the oracle like a matrix
cell (`_hold_to_oracle`, on up to 2 000 problems of the batch), the exact checker runs on a sample
and on the run's CONV_PGTOL stops, and the oracle's runs must reach the regime the option set is
meant to test (`assert_regime`).  The build that ran is asserted through `dart_se3mpc_kernel_info`.

The register-capped builds (l8_occ3, l8_b64, l16_occ3, l32_occ3, l6_occ5) store the first two
correction pairs through exact-size copies of the pair code.  Each of their runs is repeated in the
build's latency sibling (l8, l8, l16, l32, l6) on the same batch.  At the reference's settings
(modes 0 and 2, tolerance 5e-2) the two must agree as in test_gpu_build_variants_agree: identical
counters and tasks, x within 1e-11.  That rule is too strict for the long solves of the other
settings, where the separate compilations' last-bit differences grow over up to 50 iterations.
Measured on one B200 at its 1000 W limit (every option set, cold and warm): x differed by up to
4e-6 with identical counters (l8_occ3, mode 1, tolerance 1e-7, max_corrections 1), and counters
differed on up to 13 of 1 001 problems (l6_occ5, mode 0 long solves, max_corrections 1).  There the rule is the
north-star one between the builds: equal counters and tasks on at least 98 % of the batch, and on
those, x within 1e-4 and cost within 1e-5 (relative) for 99.5 %.  A build that stores a pair
wrongly misses it by far: on the host builds at max_corrections 1, the register-capped policy
with the two-pair copy taken for a one-slot ring had equal counters on 8 to 34 % of the problems
in modes 1, 3 and 4, and x off by up to 0.2 with equal counters in modes 0 and 2.

In those long solves an FTOL stop determines x to a few 1e-5 only: the oracle's own result moves
beyond 1e-4, with equal counters, after a one-ulp move of its inputs.  There a run that misses
the mode's rule passes only where the oracle against itself after one ulp misses it too, and the
run agrees with the oracle as well as the oracle agrees with itself (`_hold_to_oracle` keeps the
rule's condition on problems with equal counters; these settings drop it).

Left out to bound the run time: on the latency builds other than l8 (l4, l16, l32, l32x2, l6)
only the sets `m1` and `fun` run; the sets `m2`, `ls`, `it0` and `mix` run on l8 and on the five
capped builds.

Two routes reach a capped build without DART_SE3MPC_VARIANT, both with max_corrections 1:
`ClosedLoopSim.run(1, parts=2)` (two sub-populations of 4 096 drones, which the in-flight hint
sends to l8_occ3), checked step by step against the oracle from the GPU's own state; and the
chunked host entry at 65 541 problems.  `-s` prints the table of the runs."""
import ctypes as C

import numpy as np
import pytest

import exact_check as xc
import rollout_oracle
from edge_world import EDGE_FREE, EDGE_W, edge_cells, edge_inputs, exact_grid, oracle_grid, stationary_warm
from test_gpu_kernel_matrix import (BUILDS, EXACT_SAMPLE, ORACLE_SAMPLE, ROLLOUT_BUILDS, _agreement,
                                    _hold_to_oracle, _kernel_info, _Sub, fingerprints, gpu_grid)  # noqa: F401 (fixture)
from test_solver_options import OPTION_SETS, assert_regime, settings

pytestmark = pytest.mark.gpu

CAPPED = {5: 1, 6: 1, 7: 2, 8: 3, 10: 9}          # register-capped build -> its latency sibling
FULL = set(CAPPED) | {1}                           # builds that run every option set
REDUCED = ("m1", "fun")


def _sets(build):
    return list(OPTION_SETS) if build in FULL else list(REDUCED)


CELLS = [(b, m, s) for m in (0, 1, 2) for b in BUILDS for s in _sets(b)] + \
        [(b, m, s) for m in (3, 4) for b in ROLLOUT_BUILDS for s in _sets(b)]
_RAN = []


@pytest.fixture(scope="module")
def table():
    yield _RAN
    lines = ["", f"{'build':<10}{'mode':>5}  {'set':<5}{'setting':<7}{'options':<34}{'start':<6}{'N':>4}{'B':>7}"
                 f"{'ok':>8}{'same':>8}  {'rule':<8}{'pgtol':>6}  {'sibling':<22}tasks"]
    for r in _RAN:
        lines.append(f"{r['build']:<10}{r['mode']:>5}  {r['set']:<5}{r['setting']:<7}{r['opts']:<34}{r['start']:<6}"
                     f"{r['N']:>4}{r['B']:>7}{r['ok']:>8.4f}{r['same']:>8.4f}  {r['rule']:<8}{r['pgtol']:>6}  "
                     f"{r['sibling']:<22}{r['tasks']}")
    lines.append(f"{len(_RAN)} runs, {sum(r['rule'] == 'one-ulp' for r in _RAN)} under the one-ulp rule")
    print("\n".join(lines))


def _params(mode, N, cfg, opts):
    import dart_planner_b200 as dp
    from dart_planner_b200.config import make_params
    cfg, opts = dict(cfg), dict(opts)
    if "max_iterations" in opts:
        cfg["max_iterations"] = opts.pop("max_iterations")
    c = dp.SE3MPCConfig(prediction_horizon=N, dt=0.1, obstacle_weight=EDGE_W, **cfg)
    return make_params(c, gradient_mode=mode, obstacle_free_level=EDGE_FREE, **opts)


def _oracle(oracle_mod, mode, N, cfg, opts, p0, v0, goal, hg, x_warm=None, og=None):
    op = oracle_mod.make_params(horizon=N, dt=0.1, consistent_gradient=int(mode == 1), **dict(cfg, **opts))
    kw = dict(grid=og, obstacle_weight=EDGE_W, free_level=EDGE_FREE) if mode in (2, 4) else {}
    solve = rollout_oracle.solve_batch if mode >= 3 else oracle_mod.solve_batch
    return solve(op, p0, v0, goal, has_goal=hg, x_warm=x_warm, nthreads=16, **kw)


def _solve_gpu(params, p0, v0, goal, hg, x_warm, grid):
    from dart_planner_b200.planner import BatchWorkspace
    ws = BatchWorkspace(params, len(p0), pinned=False)
    ws.set_inputs_device(p0, v0, goal)
    ws.set_has_goal(hg)
    ws.set_warm(x_warm)
    if int(params.gradient_mode) in (2, 4):
        ws.set_map(None, penalty_grid=grid)
    return ws.solve_device().numpy()


def _use_build(monkeypatch, fingerprints, build, params, B, force=False):
    """Route the launcher to `build` (its batch size, or DART_SE3MPC_VARIANT; always the variant
    with force) and assert it."""
    variant = str(build) if force else BUILDS[build][7]
    monkeypatch.delenv("DART_SE3MPC_VARIANT", raising=False)
    if variant is not None:
        monkeypatch.setenv("DART_SE3MPC_VARIANT", variant)
    info = _kernel_info(params, B)
    assert info == fingerprints[build], f"{BUILDS[build][0]} B={B}: kernel_info {info}, the build's {fingerprints[build]}"


def _assert_same_as_sibling(got, sib, what, strict):
    """strict: test_gpu_build_variants_agree (identical counters and tasks, x within 1e-11);
    otherwise the north-star rule between the builds (module docstring).  Returns the table entry."""
    same = np.ones(len(got.x), bool)
    for k in ("nit", "nfev", "status", "task"):
        same &= np.asarray(getattr(got, k)) == np.asarray(getattr(sib, k))
    dx = np.abs(np.asarray(got.x) - np.asarray(sib.x)).max(axis=1)
    relf = np.abs(got.cost - sib.cost) / np.maximum(np.abs(sib.cost), 1.0)
    dmax = dx[same].max(initial=0.0)
    if strict:
        assert same.all(), f"{what}: counters differ from the latency sibling on {(~same).sum()} problems, " \
                           f"first {np.where(~same)[0][:5]}"
        assert dmax <= 1e-11, f"{what}: x differs from the latency sibling by {dmax:.3g}"
    else:
        assert same.mean() >= 0.98, f"{what}: counters agree with the latency sibling on {same.mean():.4f}"
        close = (dx[same] <= 1e-4) & (relf[same] <= 1e-5)
        assert close.mean() >= 0.995, f"{what}: {(~close).sum()} problems with equal counters beyond 1e-4"
    return f"{(~same).sum()} differ, dx {dmax:.1e}"


def _hold(mode, warm, got, ref, rerun, what, strict):
    """`_hold_to_oracle` at the reference's settings; in the long solves the same without its
    condition on problems with equal counters (module docstring)."""
    if strict:
        return _hold_to_oracle(mode, warm, got, ref, rerun, what)
    passes, ok, same, _ = _agreement(mode, warm, got, ref)
    if passes:
        return ok, same, False
    alt_passes, ok2, same2, _ = _agreement(mode, warm, rerun(), ref)
    assert not alt_passes, (f"{what}: misses the mode's rule (ok {ok:.4f} same {same:.4f}) where the oracle meets "
                            f"it against itself after one ulp (ok {ok2:.4f} same {same2:.4f})")
    slack = 2.0 / np.sqrt(len(ref.cost))
    assert ok >= ok2 - 0.03 - slack and same >= same2 - 0.06 - slack, \
        f"{what}: ok {ok:.4f} same {same:.4f}; the oracle against itself after one ulp: ok {ok2:.4f} same {same2:.4f}"
    return ok, same, True


@pytest.mark.parametrize("build,mode,name", CELLS, ids=[f"{BUILDS[b][0]}-mode{m}-{s}" for b, m, s in CELLS])
def test_options_cell_matches_the_oracle(oracle_mod, monkeypatch, fingerprints, table, build, mode, name):
    bname, lanes, tpl, block, minb, Ns, B, variant = BUILDS[build]
    N = Ns[0]
    cells = edge_cells("float32") if mode in (2, 4) else None
    grid, og, eg = (gpu_grid(cells), oracle_grid(oracle_mod, cells), exact_grid(cells)) if cells is not None \
        else (None, None, None)
    sub = np.arange(B) if B <= 3000 else np.unique(np.r_[np.arange(0, B, max(1, B // ORACLE_SAMPLE)), B - 1])
    hg = (np.arange(B) % 11 != 3).astype(np.uint8)
    runs = []
    for opts in OPTION_SETS[name]:
        merged = []
        for label, cfg in settings(mode):
            params = _params(mode, N, cfg, opts)
            seed = 1000 * build + 10 * mode + N
            p0, v0, goal = edge_inputs(B, seed=seed, at_goal=mode in (1, 3, 4))
            rng = np.random.default_rng(seed)
            xw = None
            for start in ("cold", "warm"):
                what = f"{bname} mode {mode} {label} {opts} N {N} B {B} {start}"
                _use_build(monkeypatch, fingerprints, build, params, B)
                got = _solve_gpu(params, p0, v0, goal, hg, xw, grid)
                xws = None if xw is None else xw[sub]
                ref = _oracle(oracle_mod, mode, N, cfg, opts, p0[sub], v0[sub], goal[sub], hg[sub], xws, og)
                rerun = lambda: _oracle(oracle_mod, mode, N, cfg, opts, np.nextafter(p0[sub], np.inf),  # noqa: E731,B023
                                        v0[sub], goal[sub], hg[sub],  # noqa: B023
                                        None if xws is None else np.nextafter(xws, np.inf), og)  # noqa: B023
                strict = label == "ref"
                ok, same, escaped = _hold(mode, start == "warm", _Sub(got, sub), ref, rerun, what, strict)
                pick = np.r_[rng.choice(B, EXACT_SAMPLE, replace=False), np.where(got.task == xc.TASK_PGTOL)[0][:8]]
                n_pg = xc.check_results(params, mode, p0, v0, goal, hg, got, pick, eg, EDGE_W, EDGE_FREE, what=what)
                sib = "-"
                if build in CAPPED:
                    _use_build(monkeypatch, fingerprints, CAPPED[build], params, B, force=True)
                    sib = BUILDS[CAPPED[build]][0] + ": " + _assert_same_as_sibling(
                        got, _solve_gpu(params, p0, v0, goal, hg, xw, grid), what, strict)
                _RAN.append(dict(build=bname, mode=mode, set=name, setting=label,
                                 opts=" ".join(f"{k}={v}" for k, v in opts.items()), start=start, N=N, B=B,
                                 ok=ok, same=same, rule="one-ulp" if escaped else "strict", pgtol=n_pg, sibling=sib,
                                 tasks=dict(zip(*[a.tolist() for a in np.unique(got.task, return_counts=True)]))))
                merged.append(ref)
                xw = got.x.copy()
                xw[:, 6 * N:] += rng.normal(0, 0.4, xw[:, 6 * N:].shape)      # tilted thrust history
                xw = stationary_warm(xw, goal, N)
        runs.append((opts, type("R", (), {k: np.concatenate([getattr(r, k) for r in merged])
                                          for k in ("nit", "nfev", "status", "task")})))
    assert_regime(name, mode, runs)


def _plant(p, v, x, N, dt, mass=1.5, g=9.81):
    a = x[:, 6 * N: 6 * N + 3] / mass - np.array([0, 0, g])
    return p + v * dt + 0.5 * a * dt ** 2, v + a * dt


@pytest.mark.parametrize("mode", [0, 3])
def test_closed_loop_parts_reach_the_capped_build_with_one_pair(oracle_mod, monkeypatch, fingerprints, mode):
    """ClosedLoopSim.run(1, parts=2) at 8 192 drones, N 8, max_corrections 1: the in-flight hint
    sends both 4 096-drone launches to l8_occ3.  Mode 0 warm starts through the 7-slot kernel
    (warm == 2).  Every step against the oracle from the GPU's own state."""
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.closed_loop import ClosedLoopSim
    from dart_planner_b200.config import make_params
    monkeypatch.delenv("DART_SE3MPC_VARIANT", raising=False)
    B, N, dt = 8192, 8, 0.1
    tol = 1e-3 if mode == 3 else 5e-2
    cfg = dp.SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=tol)
    params = make_params(cfg, gradient_mode=mode, max_corrections=1)
    L = _cabi.lib()
    L.dart_se3mpc_set_inflight_hint(B)
    try:
        assert _kernel_info(params, B // 2) == fingerprints[5]
    finally:
        L.dart_se3mpc_set_inflight_hint(0)
    assert _kernel_info(params, B // 2) == fingerprints[1]        # without the hint: the latency build
    rng = np.random.default_rng(70 + mode)
    p0 = rng.uniform(-10, 10, (B, 3))
    v0 = rng.uniform(-2, 2, (B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], axis=1)
    goal[:512] = p0[:512] + 0.02
    sim = ClosedLoopSim(params, B)
    sim.reset(p0, v0, goal)
    op = oracle_mod.make_params(horizon=N, dt=dt, convergence_tolerance=tol, max_corrections=1)
    solve = rollout_oracle.solve_batch if mode == 3 else oracle_mod.solve_batch
    sub = np.r_[np.arange(0, B, 4), np.arange(1, B, 97)]
    long_solves = 0
    for s in range(8):
        pg, vg = sim.positions().cpu().numpy().copy(), sim.velocities().cpu().numpy().copy()
        xg = sim.solution().cpu().numpy().copy() if s > 0 else None
        sim.run(1, parts=2)
        ref = solve(op, pg[sub], vg[sub], goal[sub], x_warm=None if xg is None else xg[sub], nthreads=16)
        meta = sim.meta[:, :B].cpu().numpy()[:, sub]
        same = (meta[0] == ref.nit) & (meta[1] == ref.nfev) & (meta[2] == ref.status)
        assert same.mean() >= 0.99, f"mode {mode} step {s}: counters agree on {same.mean():.4f}"
        xs = sim.solution().cpu().numpy()
        ex = np.abs(xs[sub] - ref.x).max(axis=1)
        relf = np.abs(sim.cost[:B].cpu().numpy()[sub] - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
        # test_gpu_closed_loop.py (mode 0), _agree of test_gpu_rollout.py (mode 3)
        assert (ex[same] <= 1e-4).mean() >= (0.995 if mode == 3 else 1.0), f"mode {mode} step {s}: x beyond 1e-4"
        assert (relf[same] <= 1e-5).mean() >= (0.999 if mode == 3 else 1.0), f"mode {mode} step {s}: cost beyond 1e-5"
        long_solves += int((ref.nit >= 3).sum())
        if mode == 0:
            # the plant step is exact arithmetic on the GPU's own first control
            p1, v1 = _plant(pg, vg, xs, N, dt)
            np.testing.assert_array_equal(sim.positions().cpu().numpy(), p1)
            np.testing.assert_array_equal(sim.velocities().cpu().numpy(), v1)
    assert long_solves > 0, "no solve stored two pairs"


def test_chunked_host_entry_with_one_pair(oracle_mod, monkeypatch, fingerprints):
    """dart_se3mpc_solve_batch_host at 65 541 problems (chunks on two streams, l8_occ3), N 8,
    max_corrections 1: the device entry's bits, and the oracle on a sample."""
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.config import make_params
    monkeypatch.delenv("DART_SE3MPC_VARIANT", raising=False)
    B, N = 65536 + 5, 8
    params = make_params(dp.SE3MPCConfig(prediction_horizon=N, dt=0.1), max_corrections=1)
    assert _kernel_info(params, B) == fingerprints[5]
    rng = np.random.default_rng(65)
    p0 = rng.uniform(-10, 10, (B, 3))
    v0 = rng.uniform(-2, 2, (B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (B, 2)), rng.uniform(3, 8, (B, 1))], axis=1)
    soa = lambda a: np.ascontiguousarray(np.asarray(a, np.float64).reshape(B, -1).T)  # noqa: E731
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    x = np.zeros((9 * N, B)); cost = np.zeros(B)
    nit = np.zeros(B, np.int32); nfev = np.zeros(B, np.int32); status = np.zeros(B, np.int32)
    rc = _cabi.lib().dart_se3mpc_solve_batch_host(C.byref(params), B, vp(soa(p0)), vp(soa(v0)), vp(soa(goal)),
                                                  None, None, vp(x), vp(cost), vp(nit), vp(nfev), vp(status),
                                                  None, None, None, None)
    assert rc == 0
    dev = _solve_gpu(params, p0, v0, goal, np.ones(B, np.uint8), None, None)
    np.testing.assert_array_equal(x.T, dev.x)
    np.testing.assert_array_equal(cost, dev.cost)
    for k, a in (("nit", nit), ("nfev", nfev), ("status", status)):
        np.testing.assert_array_equal(a, getattr(dev, k), err_msg=k)
    sub = np.r_[np.arange(0, B, 33), B - 1]
    ref = oracle_mod.solve_batch(oracle_mod.make_params(horizon=N, dt=0.1, max_corrections=1),
                                 p0[sub], v0[sub], goal[sub], nthreads=16)
    same = (nit[sub] == ref.nit) & (nfev[sub] == ref.nfev) & (status[sub] == ref.status)
    assert same.mean() == 1.0, f"counters agree on {same.mean():.4f}"
    assert (np.abs(x.T[sub] - ref.x).max(axis=1) <= 1e-4).all()
    assert ref.nit.max() >= 3                      # some solves stored a second pair
