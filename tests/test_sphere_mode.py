"""Sphere obstacle penalty (gradient_mode 5 = mode 0 + spheres, 6 = mode 3 + spheres), CPU tier: the
penalty and the modes' gradients against central differences, the kernel core (host build, every
policy) against the CPU restatement, bit-equality with the plain modes where no sphere is reached,
the C ABI's refusals, and the oracle's closed loop around spheres.  The restatement is
tests/sphere_oracle, the host build of the core in these modes tests/emu_spheres."""
import ctypes as C
import os

import numpy as np
import pytest

import emu_spheres
import sphere_exact
import sphere_oracle
from test_clearance_loop import ORIGIN, RES, one_sphere, oracle_loop, path_collides, sphere_world
from test_rollout_mode import GOAL_RADIUS, _inputs

W, MARGIN = 1000.0, 0.5


def sphere_list_on_paths(p0, v0, goal, n=20, seed=5):
    """n spheres where plans go: half on the straight start-goal segments (mode 5's cold start runs
    along them), half a short way along the initial velocity (mode 6's rollouts start there)."""
    rng = np.random.default_rng(seed)
    i = rng.choice(len(p0), n, replace=False)
    c = np.where((np.arange(n) % 2 == 0)[:, None], 0.5 * (p0[i] + goal[i]), p0[i] + 0.4 * v0[i])
    return sphere_oracle.sphere_list(c + rng.normal(0, 0.2, (n, 3)), rng.uniform(0.6, 1.6, n))


def world_list(seed=7):
    """The analytic list of the 48-sphere world of test_rollout_mode._world (same draws)."""
    rng = np.random.default_rng(seed)
    return sphere_oracle.sphere_list(rng.uniform(-15, 15, (48, 3)), rng.uniform(0.8, 2.5, 48))


def _params(mode, N, dt=0.1, tol=1e-3):
    from dart_planner_b200.config import SE3MPCConfig, make_params
    return make_params(SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=tol, obstacle_weight=W),
                       gradient_mode=mode)


# ---- the term --------------------------------------------------------------------------------
def test_penalty_definition_and_core_agree():
    s = sphere_oracle.sphere_list([[0.0, 0.0, 5.0], [1.0, 2.0, 3.0]], [2.5, 1.0])
    # R = 3 for the first sphere: (3, 0, 5) is on the inflated surface (h = 0 exactly)
    P = np.array([[0.0, 0.0, 5.0], [3.0, 0.0, 5.0], [0.3, 0.1, 4.2], [1.2, 2.1, 3.3], [10.0, 10.0, 10.0]])
    f, g = sphere_oracle.penalty(s, P, W, MARGIN)
    fe, ge = emu_spheres.penalty(s, P, W, MARGIN)
    assert f.tobytes() == fe.tobytes() and g.tobytes() == ge.tobytes()   # the core computes the definition
    assert f[0] == W * 9.0 ** 2 and (g[0] == 0).all()                     # at a centre: stationary
    assert f[1] == 0.0 and (g[1] == 0).all()                              # h = 0: no term
    assert f[4] == 0.0 and np.signbit(g[4]).all()                         # unreached: -0, the identity
    e = P[2] - s[0, :3]
    h = 9.0 - e @ e
    assert f[2] == pytest.approx(W * h * h) and g[2] == pytest.approx(-4 * W * h * e)
    assert f[3] > 0 and (g[3] != 0).all()                                 # inside both spheres


@pytest.mark.parametrize("N", [1, 6, 8])
@pytest.mark.parametrize("mode", [5, 6])
def test_gradient_matches_central_differences(oracle_mod, mode, N):
    op = oracle_mod.make_params(horizon=N, dt=0.1)
    rng = np.random.default_rng(N + 10 * mode)
    for trial in range(6):
        p0, v0 = rng.uniform(-3, 3, 3), rng.uniform(-2, 2, 3)
        goal = None if trial == 5 else rng.uniform(-5, 5, 3)
        T = rng.normal(0, 2, (N, 3)) + [0.0, 0.0, 14.715]
        if mode == 5:
            x = np.concatenate([p0 + rng.normal(0, 1, (N, 3)).cumsum(0), rng.normal(0, 1, (N, 3)), T]).ravel()
            Pk = x[:3 * N].reshape(N, 3)
            v = x
        else:
            Pk = sphere_oracle_rollout(op, p0, v0, T)
            v = T.ravel()
        # spheres around the positions: one inside (not at a centre), one centred on a position,
        # one with a position on its inflated surface, one out of reach
        k = rng.integers(N)
        s = [[*(Pk[k] + [0.4, -0.3, 0.2]), 1.5], [*Pk[(k + 1) % N], 0.7], [*(Pk[(k + 2) % N] - [1.25, 0.0, 0.0]), 0.75],
             [50.0, 50.0, 50.0, 1.0]]
        f, g = sphere_oracle.fg(op, mode, p0, v0, goal, v, s, W, MARGIN)
        h = 1e-6
        num = np.array([(sphere_oracle.fg(op, mode, p0, v0, goal, v + h * e, s, W, MARGIN)[0]
                         - sphere_oracle.fg(op, mode, p0, v0, goal, v - h * e, s, W, MARGIN)[0]) / (2 * h)
                        for e in np.eye(len(v))])
        tol = 1e-5 * max(np.abs(g).max(), 1.0) + 8 * 2.2e-16 * abs(f) / h
        if mode == 5:   # mode 0's gradient is the reference's (inconsistent by design): compare P only
            num, g = num[:3 * N], g[:3 * N] - sphere_oracle.fg(op, mode, p0, v0, goal, v, [], W, MARGIN)[1][:3 * N]
            num = num - np.array([(sphere_oracle.fg(op, mode, p0, v0, goal, v + h * e, [], W, MARGIN)[0]
                                   - sphere_oracle.fg(op, mode, p0, v0, goal, v - h * e, [], W, MARGIN)[0]) / (2 * h)
                                  for e in np.eye(len(v))])[:3 * N]
        assert np.abs(num - g).max() <= tol, (trial, np.abs(num - g).max(), tol)


def sphere_oracle_rollout(op, p0, v0, T):
    import rollout_oracle
    N = op.horizon
    return rollout_oracle.rollout(op, p0, v0, T)[:3 * N].reshape(N, 3)


# ---- the core against the restatement ----------------------------------------------------------
def _agree(got, ref, mode):
    same = (got.nit == ref.nit) & (got.nfev == ref.nfev) & (got.status == ref.status)
    dx = np.abs(got.x - ref.x).max(axis=1)
    relf = np.abs(got.cost - ref.cost) / np.maximum(np.abs(ref.cost), 1.0)
    lim = 1e-6 if mode == 5 else 1e-4
    return same, (dx <= lim) & (relf <= (1e-9 if mode == 5 else 1e-5))


def _hold(got, ref, mode, rerun, what):
    """The rule of the mode (tests/test_core_emulation.py for mode 2, tests/test_rollout_mode.py for
    mode 3): counters equal on nearly every problem, and x and cost close where they are.  Where it
    fails, the core must agree with the oracle as well as the oracle agrees with itself after a one-ulp
    move of the start (the escape of tests/test_gpu_kernel_matrix.py)."""
    same, close = _agree(got, ref, mode)
    need = 0.995 if mode == 5 else 0.999
    ok = same.mean() >= need and close[same].mean() >= (1.0 if mode == 5 else 0.995)
    if ok:
        return
    ref2 = rerun()
    same2, close2 = _agree(ref2, ref, mode)
    assert same.mean() >= same2.mean() - 0.005 and (same & close).mean() >= (same2 & close2).mean() - 0.005, \
        f"{what}: same {same.mean():.4f} ok {(same & close).mean():.4f}; oracle vs itself after one ulp: " \
        f"same {same2.mean():.4f} ok {(same2 & close2).mean():.4f}"


@pytest.mark.parametrize("mode,policy", [(5, p) for p in emu_spheres.POLICIES[5]] +
                         [(6, p) for p in emu_spheres.POLICIES[6]])
def test_core_matches_oracle(oracle_mod, mode, policy):
    p0, v0, goal, hg = _inputs(1500)
    s = sphere_list_on_paths(p0, v0, goal)
    emu_spheres.set_policy(policy)
    try:
        for N in (6, 8):
            op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
            pr = _params(mode, N)
            xw, pp = None, p0
            for warm in (False, True):   # cold, then warm from the cold solution at a shifted start
                run = lambda q: sphere_oracle.solve_batch(op, mode, q, v0, goal, s, W, MARGIN, has_goal=hg,  # noqa
                                                          x_warm=xw, nthreads=8)
                ref = run(pp)
                got = emu_spheres.solve_batch(pr, pp, v0, goal, s, MARGIN, has_goal=hg, x_warm=xw)
                _hold(got, ref, mode, lambda: run(np.nextafter(pp, np.inf)), f"mode {mode} {policy} N {N} warm {warm}")
                if mode == 5:
                    assert (got.x[:, 6 * N:].reshape(-1, N, 3)[..., :2] == 0).all()   # lateral thrust stays 0
                xw, pp = ref.x, pp + 0.1
    finally:
        emu_spheres.set_policy("latency")


def test_the_spheres_change_the_plans(oracle_mod):
    """The list of the tests above is reached: a good share of plans differ from the plain modes'."""
    import rollout_oracle
    p0, v0, goal, hg = _inputs(600)
    s = sphere_list_on_paths(p0, v0, goal)
    op = oracle_mod.make_params(horizon=8, dt=0.1, convergence_tolerance=1e-3)
    for mode, plain in ((5, oracle_mod.solve_batch(op, p0, v0, goal, has_goal=hg, nthreads=8)),
                        (6, rollout_oracle.solve_batch(op, p0, v0, goal, has_goal=hg, nthreads=8))):
        r = sphere_oracle.solve_batch(op, mode, p0, v0, goal, s, W, MARGIN, has_goal=hg, nthreads=8)
        assert (np.abs(r.x - plain.x).max(axis=1) > 1e-6).mean() >= 0.1, mode
        # the exact checker on the restatement's own results; the reference's tolerance 5e-2 gives
        # projected-gradient stops for check (c)
        n = 0
        for tol in (1e-3, 5e-2):
            o2 = oracle_mod.make_params(horizon=8, dt=0.1, convergence_tolerance=tol)
            r = sphere_oracle.solve_batch(o2, mode, p0, v0, goal, s, W, MARGIN, has_goal=hg, nthreads=8)
            n += sphere_exact.check_results(_params(mode, 8, tol=tol), mode, p0, v0, goal, hg, r, range(0, 600, 15),
                                            s, W, MARGIN, what=f"oracle mode {mode} tol {tol}")
        # (cold starts of mode 0 / 5 stop on the projected gradient only with the hover thrust on its
        # bound, tests/test_gpu_kernel_matrix.py: mode 5 is checked by (a) alone here)
        assert n > 0 or mode == 5, mode


# ---- unreachable spheres: the plain modes' bits --------------------------------------------------
@pytest.mark.parametrize("mode,policy", [(5, p) for p in emu_spheres.POLICIES[5]] +
                         [(6, p) for p in emu_spheres.POLICIES[6]])
def test_unreachable_spheres_give_the_plain_bits(oracle_mod, mode, policy):
    """Every position gets a penalty of +0 and a gradient of -0, the identity of the sums it enters,
    so modes 5 / 6 return exactly the bits of modes 0 / 3 -- signed zeros included."""
    import emu
    import emu_rollout
    import rollout_oracle
    p0, v0, goal, hg = _inputs(300)
    far = sphere_oracle.sphere_list([[500.0, 500.0, 500.0], [-400.0, 0.0, 0.0]], [1.0, 2.0])
    for N in (6, 8):
        op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
        pr, pp = _params(0 if mode == 5 else 3, N), _params(mode, N)
        emu_spheres.set_policy(policy)
        try:
            xw = None
            for _ in range(2):
                for s in (far, np.zeros((0, 4))):
                    got = emu_spheres.solve_batch(pp, p0, v0, goal, s, MARGIN, has_goal=hg, x_warm=xw)
                    if mode == 5:
                        emu.lib().emu_set_ls_shared(1 if policy in ("throughput", "two-phase") else 0)
                        emu.lib().emu_set_two_phase(1 if policy == "two-phase" else 0)
                        emu.lib().emu_set_cold_special(1 if policy == "seven-slot" else 0)
                        plain = emu.solve_batch(pr, p0, v0, goal, has_goal=hg, x_warm=xw)
                        ref = oracle_mod.solve_batch(op, p0, v0, goal, has_goal=hg, x_warm=xw, nthreads=8)
                    else:
                        emu_rollout.set_policy(policy)
                        plain = emu_rollout.solve_batch(pr, p0, v0, goal, has_goal=hg, x_warm=xw)
                        ref = rollout_oracle.solve_batch(op, p0, v0, goal, has_goal=hg, x_warm=xw, nthreads=8)
                    if policy == "seven-slot" and xw is not None:
                        continue   # tests/emu runs its 7-slot instantiation for cold starts only
                    for a in ("x", "cost", "nit", "nfev", "status", "task", "attitudes", "body_rates"):
                        assert getattr(got, a).tobytes() == getattr(plain, a).tobytes(), (N, a, len(s))
                    rs = sphere_oracle.solve_batch(op, mode, p0, v0, goal, s, W, MARGIN, has_goal=hg, x_warm=xw,
                                                   nthreads=8)
                    for a in ("x", "cost", "nit", "nfev", "status", "task"):
                        assert getattr(rs, a).tobytes() == getattr(ref, a).tobytes(), (N, a, len(s))
                xw = ref.x
        finally:
            emu_spheres.set_policy("latency")
            emu.lib().emu_set_ls_shared(0)
            emu.lib().emu_set_two_phase(0)
            emu.lib().emu_set_cold_special(0)
            emu_rollout.set_policy("latency")


# ---- the C ABI's refusals (no GPU needed: they come before any CUDA call) -------------------------
def test_sphere_entries_refuse_bad_arguments_without_a_gpu():
    from dart_planner_b200 import _cabi
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("library not built")
    L = _cabi.lib()
    OK, BAD, UNS = _cabi.DART_OK, _cabi.DART_E_BADARG, _cabi.DART_E_UNSUPPORTED
    buf = np.zeros(64 * 9 * 4)
    bp = buf.ctypes.data
    lst = np.zeros((2, 4))
    sph = _cabi.Spheres(2, 0, lst.ctypes.data, 0.5)

    def p(mode, N=8):
        q = _params(0, N)
        q.gradient_mode = mode
        return q

    def dev(q, s, B=0):
        return L.dart_se3mpc_solve_batch_spheres(C.byref(q), B, B, bp, bp, bp, *([None] * 13),
                                                 None if s is None else C.byref(s), None, 0.0, 0.0, None, None)

    def host(q, s, B=0):
        return L.dart_se3mpc_solve_batch_host_spheres(C.byref(q), B, bp, bp, bp, *([None] * 11),
                                                      None if s is None else C.byref(s))

    def loop(q, s, warm=1, B=0):
        return L.dart_se3mpc_closed_loop_step_spheres(C.byref(q), B, B, bp, bp, bp, None, bp, warm, None, None, None,
                                                      None, 0.1, None if s is None else C.byref(s), None, 0.0, 0.6, 0,
                                                      None, None)

    for call in (dev, host, loop):
        assert call(p(5), sph) == OK and call(p(6), sph) == OK
        for mode in (0, 1, 2, 3, 4, 7, -1):
            assert call(p(mode), sph) == BAD, (call.__name__, mode)
        assert call(p(5), None) == BAD
        assert call(p(5), _cabi.Spheres(-1, 0, lst.ctypes.data, 0.5)) == BAD
        assert call(p(6), _cabi.Spheres(3, 0, None, 0.5)) == BAD
        assert call(p(5), _cabi.Spheres(0, 0, None, 0.5)) == OK          # an empty list
        assert call(p(6, 17), sph) == UNS and call(p(6, 16), sph) == OK
        assert call(p(5, 64), sph) == OK and call(p(5, 65), sph) == UNS  # mode 5: every horizon
    assert loop(p(6), sph, warm=2) == BAD and loop(p(5), sph, warm=2) == OK
    # the existing entries keep refusing the new modes
    for mode in (5, 6):
        q = p(mode)
        assert L.dart_se3mpc_solve_batch(C.byref(q), 0, 0, bp, bp, bp, *([None] * 14)) == UNS
        assert L.dart_se3mpc_solve_batch_map(C.byref(q), 0, 0, bp, bp, bp, *([None] * 13), None, 0.0, 0.0,
                                             None, None) == UNS
        assert L.dart_se3mpc_solve_batch_host(C.byref(q), 0, bp, bp, bp, *([None] * 11)) == UNS
        assert L.dart_se3mpc_closed_loop_step(C.byref(q), 0, 0, bp, bp, bp, None, bp, 1, None, None, None, None,
                                              0.1, None) == UNS
        assert L.dart_se3mpc_closed_loop_step_map(C.byref(q), 0, 0, bp, bp, bp, None, bp, 1, None, None, None,
                                                  None, 0.1, None, None, 0.0, 0.6, 0, None, None) == UNS
        assert L.dart_se3mpc_solve_batch_rows(C.byref(q), 0, 0, bp, bp, bp, None, None, None, bp, 64, 0, None,
                                              0.0, 0.0, 0, None) == UNS
        assert L.dart_se3mpc_kernel_info(C.byref(q), 1, None, None, None, None, None) == UNS


def test_python_refusals_without_a_gpu():
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.closed_loop import ClosedLoopSim
    s = (np.zeros((1, 3)), np.ones(1))
    with pytest.raises(ValueError, match="obstacle_penalty"):
        dp.plan_batch(np.zeros((2, 3)), np.zeros((2, 3)), np.ones((2, 3)), spheres=s, obstacle_penalty=True)
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("library not built")
    with pytest.raises(ValueError, match="spheres"):
        ClosedLoopSim(_params(5, 8), 4)
    with pytest.raises(ValueError, match="spheres"):
        ClosedLoopSim(_params(0, 8), 4, spheres=s)


# ---- the oracle's closed loop around the spheres --------------------------------------------------
def sphere_loop(og, p0, goal, spheres, margin, steps=100, N=8, dt=0.1, tol=1e-3):
    """oracle_loop (test_clearance_loop) in mode 6 with the analytic sphere list."""
    import oracle
    op = oracle.make_params(horizon=N, dt=dt, convergence_tolerance=tol)
    p, v, x = p0.copy(), np.zeros_like(p0), None
    first = np.full(len(p0), -1)
    for s in range(steps):
        x = sphere_oracle.solve_batch(op, 6, p, v, goal, spheres, W, margin, x_warm=x, nthreads=16).x
        pn, v = x[:, 3:6].copy(), x[:, 3 * N + 3:3 * N + 6].copy()
        hit = path_collides(og.occ, ORIGIN, RES, og.g.prior, p, pn, 0.0, 0.6)
        first[hit & (first < 0)] = s
        p = pn
    return first, p


# Measured (N 8, dt 0.1, tolerance 1e-3, 100 replans, w 1000, margin 1 m, collisions judged on the
# rasterised map): one sphere, 128 crossing drones: mode 3 126 / 128 (98.4 %), mode 6 0; the
# 48-sphere world, 256 drones: mode 3 24 / 256 (9.4 %), mode 6 1 / 256 (0.39 %).  Every mode-6 drone
# ends within 3.2e-6 m of its goal.  (With margin 0.5 m, 20 % and 3.5 % collide: the rasterised
# spheres are larger than the analytic ones by up to a voxel diagonal, 0.69 m.)
@pytest.mark.parametrize("scenario", ["one_sphere", "sphere_world"])
def test_oracle_loop_around_spheres(oracle_mod, scenario):
    if scenario == "one_sphere":
        og, p0, goal = one_sphere(oracle_mod)
        spheres = sphere_oracle.sphere_list([[0.0, 0.0, 5.0]], [2.5])
    else:
        og, p0, goal = sphere_world(oracle_mod)
        spheres = world_list()
    first3, _ = oracle_loop(oracle_mod, og, p0, goal)
    first6, p = sphere_loop(og, p0, goal, spheres, 1.0)
    frac3, frac6 = (first3 >= 0).mean(), (first6 >= 0).mean()
    assert frac6 < frac3, (frac6, frac3)
    assert (frac3, frac6) == ((126 / 128, 0.0) if scenario == "one_sphere" else (24 / 256, 1 / 256))
    assert np.linalg.norm(p - goal, axis=1).max() <= GOAL_RADIUS
