"""SciPy's L-BFGS-B options (max_corrections, max_linesearch, max_fun, max_iterations) away from
their defaults: the kernel core (host builds tests/emu and tests/emu_rollout) against the oracles,
and every build policy against every other, on the CPU tier.

The policies run different copies of the stored-pair code: the register-capped and two-phase
policies store the first and second pair through exact-size copies (se3mpc_core.cuh, ringc), the
register-rich policy through the general ring code.  The arithmetic of the copies is the same, so
every policy must return the same bits.  A copy taken where it does not apply -- the two-pair copy
with a correction memory of one -- silently solves another problem, which the oracle rule alone
catches only at some option sets.

Each option set is checked to reach the regime it is meant to test (`assert_regime`), so that a set
which stops doing so fails instead of passing empty.  tests/test_gpu_solver_options.py uses the
same sets and checks on the GPU."""
import numpy as np
import pytest

import rollout_oracle
from conftest import COST_RTOL, CTRL_ATOL

# name -> the option runs of the set (keyword arguments of make_params)
OPTION_SETS = {
    "m1": [dict(max_corrections=1)],
    "m2": [dict(max_corrections=2)],
    "ls": [dict(max_linesearch=1), dict(max_linesearch=2)],
    "fun": [dict(max_fun=3), dict(max_fun=8)],
    "it0": [dict(max_iterations=0)],
    "mix": [dict(max_corrections=1, max_linesearch=2, max_fun=5)],
}
TASK_PGTOL, TASK_FTOL, TASK_MAXITER, TASK_MAXFUN, TASK_ABNORMAL = 1, 2, 3, 4, 5
OBSTACLE_W = 1000.0


def settings(mode):
    """The solver settings each option set runs at in a mode: (label, SE3MPCConfig overrides).  The
    modes with the reference gradient (0, 2) run the reference's settings ("ref"), where solves end
    within three iterations, and longer solves that store more pairs: small position and velocity
    weights at tolerance 1e-5 in mode 0 (test_core_emulation.py), tolerance 1e-3 in mode 2.  The
    modes with an exact gradient (1, 3, 4) run long solves at tolerance 1e-7."""
    if mode == 0:
        return [("ref", dict(convergence_tolerance=5e-2, max_iterations=15)),
                ("long", dict(position_weight=3.0, velocity_weight=0.1, convergence_tolerance=1e-5,
                              max_iterations=50))]
    if mode == 2:
        return [("ref", dict(convergence_tolerance=5e-2, max_iterations=15)),
                ("long", dict(convergence_tolerance=1e-3, max_iterations=15))]
    return [("tight", dict(convergence_tolerance=1e-7, max_iterations=30))]


def oracle_params(oracle_mod, mode, N, dt, cfg, opts):
    return oracle_mod.make_params(horizon=N, dt=dt, consistent_gradient=int(mode == 1), **dict(cfg, **opts))


def lib_params(mode, N, dt, cfg, opts):
    from dart_planner_b200.config import SE3MPCConfig, make_params
    cfg = dict(cfg, obstacle_weight=OBSTACLE_W)
    opts = dict(opts)
    if "max_iterations" in opts:
        cfg["max_iterations"] = opts.pop("max_iterations")
    return make_params(SE3MPCConfig(prediction_horizon=N, dt=dt, **cfg), gradient_mode=mode, **opts)


def assert_regime(name, mode, runs):
    """The oracle's own runs of an option set reach the regime the set is meant to test.  runs: a
    list of (options, result with nit, nfev, status, task), the results of one option run merged."""
    what = f"option set {name} mode {mode}"
    nit = np.concatenate([r.nit for _, r in runs])
    task = np.concatenate([r.task for _, r in runs])
    tasks = sorted(set(task.tolist()))
    if name == "m1":
        # two pairs or more stored, so the second replaced the first in the one slot
        assert nit.max() >= (3 if mode in (0, 2) else 6), (what, nit.max())
    elif name == "m2":
        # the two-slot ring wraps at the third pair, moving its head to 1, and back at the fourth
        assert nit.max() >= 4, (what, nit.max())
    elif name == "ls":
        # a line search ran out of trial points with no pair stored
        assert TASK_ABNORMAL in tasks, (what, tasks)
    elif name == "fun":
        # the evaluation budget stops solves (short horizons may finish within the larger budget)
        assert TASK_MAXFUN in tasks, (what, tasks)
        for opts, r in runs:
            hit = r.task == TASK_MAXFUN
            assert (r.status[hit] == 1).all() and (r.nfev[hit] > opts["max_fun"]).all(), (what, opts)
    elif name == "it0":
        # every solve ends after its first iteration (STOP_MAXITER, nit 1), unless it ends before:
        # a start that is already stationary (CONV_PGTOL, nit 0), or a first line search that fails
        # (ABNORMAL, nit 0: the reference gradient, the occupancy penalty's kinks)
        first = (task == TASK_MAXITER) & (nit == 1)
        before = ((task == TASK_PGTOL) | (task == TASK_ABNORMAL)) & (nit == 0)
        assert (first | before).all() and first.mean() > 0.5, (what, tasks, sorted(set(nit.tolist())))
        status = np.concatenate([r.status for _, r in runs])
        assert (status[first] == 1).all(), what
    elif name == "mix":
        assert nit.max() >= 3 and TASK_MAXFUN in tasks, (what, nit.max(), tasks)
    else:
        raise AssertionError(f"unknown option set {name}")


def counters_equal(got, ref):
    return (got.nit == ref.nit) & (got.nfev == ref.nfev) & (got.status == ref.status)


def _rule(mode, got, ref):
    """(passes, fraction ok, fraction same, same_ok): the suite's rule for the mode; same_ok is its
    condition on the problems with equal counters, which here includes an equal task.  Modes 3/4:
    test_rollout_mode.py.  Modes 0-2: the fractions of test_core_emulation.py, with the north-star
    tolerance on the problems with equal counters (test_gpu_parity.py, test_gpu_config3.py): at
    tolerance 1e-7 and in the long solves, an FTOL stop determines x to a few 1e-5 only, and the
    oracle's own result moves that far, with equal counters, after a one-ulp move of its inputs."""
    same = counters_equal(got, ref)
    dx = np.abs(got.x - ref.x).max(axis=1)
    relf = np.abs(got.cost - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
    ok = (relf <= COST_RTOL) & (dx <= CTRL_ATOL)
    same_ok = bool((got.task[same] == ref.task[same]).all())
    if mode >= 3:
        frac = 0.999
        same_ok = same_ok and (dx[same] <= 1e-4).mean() >= 0.995 and bool((relf[same] <= 1e-5).all())
    else:
        frac = 0.995 if mode == 2 else 0.99
        same_ok = same_ok and bool(ok[same].all())
    return same.mean() >= frac and same_ok, ok.mean(), same.mean(), same_ok


def assert_oracle_rule(mode, got, ref, rerun, what):
    """The mode's rule; or, where the oracle itself misses the rule against its own result after a
    one-ulp move of its inputs (rerun()), agreement as good as the oracle's with itself, with the
    rule's condition on the problems with equal counters kept (test_gpu_kernel_matrix.py)."""
    passes, ok, same, same_ok = _rule(mode, got, ref)
    if passes:
        return
    assert same_ok, f"{what}: out of tolerance, or another task, with equal counters (ok {ok:.4f} same {same:.4f})"
    alt_passes, ok2, same2, _ = _rule(mode, rerun(), ref)
    assert not alt_passes, (f"{what}: misses the mode's rule (ok {ok:.4f} same {same:.4f}) where the oracle meets "
                            f"it against itself after one ulp (ok {ok2:.4f} same {same2:.4f})")
    slack = 2.0 / np.sqrt(len(ref.cost))
    assert ok >= ok2 - 0.03 - slack and same >= same2 - 0.06 - slack, \
        f"{what}: ok {ok:.4f} same {same:.4f}; the oracle against itself after one ulp: ok {ok2:.4f} same {same2:.4f}"


COUNTERS = ("nit", "nfev", "status", "task")
FIELDS = ("x", "cost") + COUNTERS


def assert_bit_identical(got, base, what):
    for k in FIELDS:
        a, b = getattr(got, k), getattr(base, k)
        bad = np.where((a != b).reshape(len(a), -1).any(axis=1))[0]
        assert bad.size == 0, f"{what}: {k} differs from the register-rich policy on {bad.size} of {len(a)} problems, " \
                              f"first {bad[:5]}"


def _inputs(B, seed):
    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-5, 5, (B, 3))
    v0 = rng.uniform(-2, 2, (B, 3))
    goal = rng.uniform(-5, 5, (B, 3))
    hg = (np.arange(B) % 13 != 5).astype(np.uint8)
    return p0, v0, goal, hg


def _tilted(x, N, seed):
    xw = x.copy()
    xw[:, 6 * N:] += np.random.default_rng(seed).normal(0, 0.4, xw[:, 6 * N:].shape)
    return xw


def _world(oracle_mod):
    rng = np.random.default_rng(7)
    og = oracle_mod.DenseGrid((64, 64, 64), (-32, -32, -32), 0.4)
    for c, r in zip(rng.uniform(-6, 6, (24, 3)), rng.uniform(0.8, 2.0, 24)):
        og.add_sphere(c, r)
    return og


POLICIES = {"regs": (0, 0, 0), "capped": (1, 0, 0), "cold7": (0, 1, 0), "two-phase": (1, 0, 1),
            "two-phase-cold7": (1, 1, 1)}          # (ls_shared, cold_special, two_phase)
ROLLOUT_POLICIES = ("latency", "throughput", "two-phase")


def _emu_solve(policy, pr, p0, v0, goal, hg, xw, grid):
    import emu
    L = emu.lib()
    ls, cold, two = POLICIES[policy]
    L.emu_set_ls_shared(ls)
    L.emu_set_cold_special(cold)
    L.emu_set_two_phase(two)
    try:
        return emu.solve_batch(pr, p0, v0, goal, has_goal=hg, x_warm=xw, grid=grid)
    finally:
        L.emu_set_ls_shared(0)
        L.emu_set_cold_special(0)
        L.emu_set_two_phase(0)


def _emr_solve(policy, pr, p0, v0, goal, hg, xw, grid):
    import emu_rollout
    emu_rollout.set_policy(policy)
    try:
        return emu_rollout.solve_batch(pr, p0, v0, goal, has_goal=hg, x_warm=xw, grid=grid)
    finally:
        emu_rollout.set_policy("latency")


def _once(f):
    memo = []
    return lambda: memo[0] if memo else memo.append(f()) or memo[0]


class _Counters:
    def __init__(self, results):
        for k in COUNTERS:
            setattr(self, k, np.concatenate([getattr(r, k) for r in results]))


@pytest.mark.parametrize("name", list(OPTION_SETS))
@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_options_every_policy_matches_the_oracle_and_each_other(oracle_mod, mode, name):
    """Every option run of the set, at every setting of the mode, N = 6 and 8, cold and then warm
    from the oracle's solution with tilted thrusts: every policy is held to the oracle rule and
    returns the register-rich policy's bits."""
    from dart_planner_b200 import _cabi
    og = _world(oracle_mod) if mode in (2, 4) else None
    grid = _cabi.Grid(64, 64, 64, -32, -32, -32, 0.4, 0.5, og.occ.ctypes.data) if og is not None else None
    okw = dict(grid=og, obstacle_weight=OBSTACLE_W, free_level=0.5) if og is not None else {}
    solve_ref = rollout_oracle.solve_batch if mode >= 3 else oracle_mod.solve_batch
    policies, solve = (ROLLOUT_POLICIES, _emr_solve) if mode >= 3 else (list(POLICIES), _emu_solve)
    dt = 0.1
    runs = []
    for opts in OPTION_SETS[name]:
        refs = []
        for label, cfg in settings(mode):
            for N, B in ((6, 192), (8, 256)):
                p0, v0, goal, hg = _inputs(B, seed=10 * mode + N)
                op = oracle_params(oracle_mod, mode, N, dt, cfg, opts)
                pr = lib_params(mode, N, dt, cfg, opts)
                xw = None
                for start in ("cold", "warm"):
                    what = f"mode {mode} {label} {opts} N {N} {start}"
                    ref = solve_ref(op, p0, v0, goal, has_goal=hg, x_warm=xw, nthreads=8, **okw)
                    rerun = _once(lambda: solve_ref(op, np.nextafter(p0, np.inf), v0, goal, has_goal=hg,  # noqa: B023
                                                    x_warm=None if xw is None else np.nextafter(xw, np.inf),  # noqa: B023
                                                    nthreads=8, **okw))
                    base = None
                    for policy in policies:
                        got = solve(policy, pr, p0, v0, goal, hg, xw, grid)
                        assert_oracle_rule(mode, got, ref, rerun, f"{what} {policy}")
                        if base is None:
                            base = got
                        else:
                            assert_bit_identical(got, base, f"{what} {policy}")
                    refs.append(ref)
                    xw = _tilted(ref.x, N, seed=N)
        runs.append((opts, _Counters(refs)))
    assert_regime(name, mode, runs)
