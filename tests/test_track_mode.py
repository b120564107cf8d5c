"""Reference tracking (gradient_mode 7 = mode 3 with a per-timestep reference, 8 = mode 6 with it),
CPU tier: the modes' gradients against central differences, the kernel core (host build, every
policy) against the CPU restatement, the bits of modes 3 / 6 when the reference is the goal at rest,
the C ABI's refusals, and the oracle's closed loop along paths.  The restatement is
tests/track_oracle, the host build of the core in these modes tests/emu_track."""
import ctypes as C
import os

import numpy as np
import pytest

import emu_track
import track_exact
import track_oracle
from test_clearance_loop import ORIGIN, RES, path_collides, sphere_world
from test_rollout_mode import _inputs
from test_sphere_mode import MARGIN, W, _hold, sphere_list_on_paths, world_list
from track_paths import circle_paths, polyline_paths, tracking_error


def _params(mode, N, dt=0.1, tol=1e-3):
    from dart_planner_b200.config import SE3MPCConfig, make_params
    return make_params(SE3MPCConfig(prediction_horizon=N, dt=dt, convergence_tolerance=tol, obstacle_weight=W),
                       gradient_mode=mode)


def random_reference(p0, N, seed, T=None):
    """A reference near the starts: a random walk of positions and random velocities, T samples."""
    rng = np.random.default_rng(seed)
    T = N if T is None else T
    P = p0[:, None] + rng.normal(0, 0.6, (len(p0), T, 3)).cumsum(1)
    V = rng.normal(0, 2, (len(p0), T, 3))
    return P, V


# ---- the gradient ------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 6, 8, 13])
@pytest.mark.parametrize("mode", [7, 8])
def test_gradient_matches_central_differences(oracle_mod, mode, N):
    op = oracle_mod.make_params(horizon=N, dt=0.1)
    rng = np.random.default_rng(N + 10 * mode)
    import rollout_oracle
    for trial in range(6):
        p0, v0 = rng.uniform(-3, 3, 3), rng.uniform(-2, 2, 3)
        T = rng.normal(0, 2, (N, 3)) + [0.0, 0.0, 14.715]
        Tr = int(rng.integers(1, N + 4))                     # shorter and longer than the horizon
        start = int(rng.integers(0, 4))
        P, V = random_reference(p0[None], N, trial, T=Tr)
        s = None
        if mode == 8:
            Pk = rollout_oracle.rollout(op, p0, v0, T)[:3 * N].reshape(N, 3)
            k = rng.integers(N)
            # inside (not at a centre), centred on a position, on the inflated surface, out of reach
            s = [[*(Pk[k] + [0.4, -0.3, 0.2]), 1.5], [*Pk[(k + 1) % N], 0.7],
                 [*(Pk[(k + 2) % N] - [1.25, 0.0, 0.0]), 0.75], [50.0, 50.0, 50.0, 1.0]]
        hg = trial != 5
        f, g = track_oracle.fg(op, mode, p0, v0, (P[0], V[0]), T, s, W, MARGIN, start=start, has_goal=hg)
        h = 1e-2 if mode == 7 else 1e-6            # mode 7 is quadratic in T: differences are exact
        num = np.array([(track_oracle.fg(op, mode, p0, v0, (P[0], V[0]), T.ravel() + h * e, s, W, MARGIN,
                                         start=start, has_goal=hg)[0]
                         - track_oracle.fg(op, mode, p0, v0, (P[0], V[0]), T.ravel() - h * e, s, W, MARGIN,
                                           start=start, has_goal=hg)[0]) / (2 * h) for e in np.eye(3 * N)])
        tol = 1e-5 * max(np.abs(g).max(), 1.0) + 8 * 2.2e-16 * abs(f) / h
        assert np.abs(num - g).max() <= tol, (trial, np.abs(num - g).max(), tol)
        # f is the definition at the rolled-out vector, restated here with the window of samples
        x = rollout_oracle.rollout(op, p0, v0, T)
        rp, rv = track_exact.window(P[0], V[0], start, N)
        Pk, Vk = x[:3 * N].reshape(N, 3), x[3 * N:6 * N].reshape(N, 3)
        wp = np.r_[np.ones(N - 1), 11.0] * (100.0 if hg else 0.0)
        a = T / 1.5 - [0.0, 0.0, 9.81]
        fr = (wp * ((Pk - rp) ** 2).sum(1)).sum() + 10 * ((Vk - rv) ** 2).sum() + (a ** 2).sum() \
            + 0.1 * ((T - [0.0, 0.0, 14.715]) ** 2).sum()
        if mode == 8:
            import sphere_oracle
            fr += sphere_oracle.penalty(np.asarray(s), Pk, W, MARGIN)[0].sum()
        assert f == pytest.approx(fr, rel=1e-12)


# ---- the core against the restatement ------------------------------------------------------------
@pytest.mark.parametrize("mode,policy", [(m, p) for m in (7, 8) for p in emu_track.POLICIES])
def test_core_matches_oracle(oracle_mod, mode, policy):
    p0, v0, goal, hg = _inputs(800)
    s = sphere_list_on_paths(p0, v0, goal) if mode == 8 else None
    emu_track.set_policy(policy)
    try:
        for N in (6, 8, 13):
            op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
            pr = _params(mode, N)
            ref = random_reference(p0, N, N, T=N + 3)
            xw, pp, start = None, p0, 0
            for warm in (False, True):   # cold, then warm from the cold solution a step along the path
                run = lambda q: track_oracle.solve_batch(op, mode, q, v0, ref, start, s, W, MARGIN,  # noqa: E731
                                                         has_goal=hg, x_warm=xw, nthreads=8)
                r0 = run(pp)
                got = emu_track.solve_batch(pr, pp, v0, ref, start, s, MARGIN, has_goal=hg, x_warm=xw)
                _hold(got, r0, 6, lambda: run(np.nextafter(pp, np.inf)), f"mode {mode} {policy} N {N} warm {warm}")
                xw, pp, start = r0.x, pp + 0.1, start + 1
    finally:
        emu_track.set_policy("latency")


def test_exact_checks_on_the_restatement(oracle_mod):
    """The exact checker on the oracle's own results, with projected-gradient stops for check (c)."""
    p0, v0, goal, hg = _inputs(300)
    v0[::8] = 0.0                                           # at rest on a reference that holds the start
    s = sphere_list_on_paths(p0, v0, goal)
    for mode in (7, 8):
        n = 0
        for tol in (1e-3, 5e-2):
            op = oracle_mod.make_params(horizon=8, dt=0.1, convergence_tolerance=tol)
            ref = random_reference(p0, 8, 3, T=10)
            ref[0][::8], ref[1][::8] = p0[::8, None], 0.0
            sm = s if mode == 8 else None
            r = track_oracle.solve_batch(op, mode, p0, v0, ref, 1, sm, W, MARGIN, has_goal=hg, nthreads=8)
            n += track_exact.check_results(_params(mode, 8, tol=tol), p0, v0, ref, 1, hg, r, range(0, 300, 10),
                                           sm, W, MARGIN, what=f"oracle mode {mode} tol {tol}")
        assert n > 0, mode


# ---- the goal at rest: the bits of modes 3 / 6 -------------------------------------------------------
@pytest.mark.parametrize("mode,policy", [(m, p) for m in (7, 8) for p in emu_track.POLICIES])
def test_goal_reference_gives_the_plain_bits(oracle_mod, mode, policy):
    """r_k = goal and u_k = +0: e and ev are mode 3's doubles, so every result is mode 3's (mode 8:
    mode 6's, with a list that plans reach and with an empty one), bit for bit."""
    import emu_rollout
    import emu_spheres
    import rollout_oracle
    import sphere_oracle
    p0, v0, goal, hg = _inputs(300)
    lists = (sphere_list_on_paths(p0, v0, goal), np.zeros((0, 4))) if mode == 8 else (None,)
    try:
        for N in (6, 8, 13):
            op = oracle_mod.make_params(horizon=N, dt=0.1, convergence_tolerance=1e-3)
            ref = (np.repeat(goal[:, None], N, 1), None)
            emu_track.set_policy(policy)
            emu_rollout.set_policy(policy)
            emu_spheres.set_policy(policy)
            for s in lists:
                xw = None
                for _ in range(2):
                    got = emu_track.solve_batch(_params(mode, N), p0, v0, ref, 0, s, MARGIN, has_goal=hg, x_warm=xw)
                    rt = track_oracle.solve_batch(op, mode, p0, v0, ref, 0, s, W, MARGIN, has_goal=hg, x_warm=xw,
                                                  nthreads=8)
                    if mode == 7:
                        plain = emu_rollout.solve_batch(_params(3, N), p0, v0, goal, has_goal=hg, x_warm=xw)
                        ref_o = rollout_oracle.solve_batch(op, p0, v0, goal, has_goal=hg, x_warm=xw, nthreads=8)
                    else:
                        plain = emu_spheres.solve_batch(_params(6, N), p0, v0, goal, s, MARGIN, has_goal=hg, x_warm=xw)
                        ref_o = sphere_oracle.solve_batch(op, 6, p0, v0, goal, s, W, MARGIN, has_goal=hg, x_warm=xw,
                                                          nthreads=8)
                    for a in ("x", "cost", "nit", "nfev", "status", "task", "attitudes", "body_rates"):
                        assert getattr(got, a).tobytes() == getattr(plain, a).tobytes(), (N, a, policy)
                    for a in ("x", "cost", "nit", "nfev", "status", "task"):
                        assert getattr(rt, a).tobytes() == getattr(ref_o, a).tobytes(), (N, a)
                    xw = ref_o.x
    finally:
        emu_track.set_policy("latency")
        emu_rollout.set_policy("latency")
        emu_spheres.set_policy("latency")


# ---- the C ABI's refusals (no GPU needed: they come before any CUDA call) -------------------------
def test_track_entries_refuse_bad_arguments_without_a_gpu():
    from dart_planner_b200 import _cabi
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("library not built")
    L = _cabi.lib()
    OK, BAD, UNS = _cabi.DART_OK, _cabi.DART_E_BADARG, _cabi.DART_E_UNSUPPORTED
    buf = np.zeros(64 * 9 * 4)
    bp = buf.ctypes.data
    lst = np.zeros((2, 4))
    sph = _cabi.Spheres(2, 0, lst.ctypes.data, 0.5)
    ref = _cabi.TrackRef(8, 0, bp)

    def p(mode, N=8):
        q = _params(0, N)
        q.gradient_mode = mode
        return q

    def dev(q, r, s, B=0):
        return L.dart_se3mpc_solve_batch_track(C.byref(q), B, B, bp, bp, *([None] * 13),
                                               None if r is None else C.byref(r), None if s is None else C.byref(s),
                                               None, 0.0, 0.0, None, None)

    def loop(q, r, s, warm=1, B=0, plant_dt=0.1):
        return L.dart_se3mpc_closed_loop_step_track(C.byref(q), B, B, bp, bp, None, bp, warm, None, None, None, None,
                                                    plant_dt, None if r is None else C.byref(r),
                                                    None if s is None else C.byref(s), None, 0.0, 0.6, 0, None, None)

    for call in (dev, loop):
        assert call(p(7), ref, None) == OK and call(p(8), ref, sph) == OK
        for mode in (0, 1, 2, 3, 4, 5, 6, 9, -1):
            assert call(p(mode), ref, None) == BAD and call(p(mode), ref, sph) == BAD, (call.__name__, mode)
        assert call(p(7), None, None) == BAD
        assert call(p(7), _cabi.TrackRef(8, 0, None), None) == BAD
        assert call(p(7), _cabi.TrackRef(0, 0, bp), None) == BAD
        assert call(p(7), _cabi.TrackRef(8, -1, bp), None) == BAD
        assert call(p(7), _cabi.TrackRef(1, 1 << 30, bp), None) == OK        # far past the end: held
        assert call(p(7), ref, sph) == BAD and call(p(8), ref, None) == BAD
        assert call(p(8), ref, _cabi.Spheres(-1, 0, lst.ctypes.data, 0.5)) == BAD
        assert call(p(8), ref, _cabi.Spheres(0, 0, None, 0.5)) == OK          # an empty list
        assert call(p(7, 17), ref, None) == UNS and call(p(7, 16), ref, None) == OK
        assert call(p(8, 17), ref, sph) == UNS and call(p(8, 1), ref, sph) == OK
    assert loop(p(7), ref, None, warm=2) == BAD and loop(p(8), ref, sph, warm=2) == BAD
    assert loop(p(7), ref, None, plant_dt=0.05) == BAD and loop(p(7), ref, None, plant_dt=0.1) == OK
    # the existing entries keep refusing the new modes
    for mode in (7, 8):
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
        assert L.dart_se3mpc_solve_batch_spheres(C.byref(q), 0, 0, bp, bp, bp, *([None] * 13), C.byref(sph), None,
                                                 0.0, 0.0, None, None) == BAD
        assert L.dart_se3mpc_solve_batch_host_spheres(C.byref(q), 0, bp, bp, bp, *([None] * 11), C.byref(sph)) == BAD
        assert L.dart_se3mpc_closed_loop_step_spheres(C.byref(q), 0, 0, bp, bp, bp, None, bp, 1, None, None, None,
                                                      None, 0.1, C.byref(sph), None, 0.0, 0.6, 0, None, None) == BAD


def test_python_refusals_without_a_gpu():
    import dart_planner_b200 as dp
    from dart_planner_b200 import _cabi
    from dart_planner_b200.closed_loop import ClosedLoopSim
    P = np.zeros((2, 8, 3))
    with pytest.raises(ValueError, match="dynamics_consistent"):
        dp.plan_batch(np.zeros((2, 3)), np.zeros((2, 3)), None, reference=(P, None))
    with pytest.raises(ValueError, match="reference"):
        dp.plan_batch(np.zeros((2, 3)), np.zeros((2, 3)), None)
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("library not built")
    with pytest.raises(ValueError, match="reference_path"):
        ClosedLoopSim(_params(7, 8), 2)
    with pytest.raises(ValueError, match="reference_path"):
        ClosedLoopSim(_params(3, 8), 2, reference_path=(P, None))
    with pytest.raises(ValueError, match="plant_dt"):
        ClosedLoopSim(_params(7, 8), 2, plant_dt=0.05, reference_path=(P, None))
    with pytest.raises(ValueError, match="spheres"):
        ClosedLoopSim(_params(8, 8), 2, reference_path=(P, None))


# ---- the oracle's closed loop along paths ---------------------------------------------------------
N_LOOP, DT, STEPS, T_PATH = 8, 0.1, 100, 60


def chase_loop(op, p0, v0, P, steps):
    """Mode 3 re-aimed at every replan ("carrot chasing"): step s flies to path sample
    min(s + N - 1, T - 1), the end of the window mode 7 tracks."""
    import rollout_oracle
    N, T = op.horizon, P.shape[1]
    pp, vv, x, hist = p0.copy(), v0.copy(), None, []
    for s in range(steps):
        x = rollout_oracle.solve_batch(op, pp, vv, P[:, min(s + N - 1, T - 1)], x_warm=x, nthreads=16).x
        pp, vv = x[:, 3:6].copy(), x[:, 3 * N + 3:3 * N + 6].copy()
        hist.append(pp)
    return np.stack(hist)


def loop_errors(hist, P):
    d = tracking_error(hist, P)[19:]          # steps 20..100: positions at times 20..100
    return float(np.sqrt((d ** 2).mean())), float(d.max())


# Measured (128 drones, N 8, dt 0.1, tolerance 1e-3, 100 replans, a 60-sample path, error = distance
# to the current path sample over times 20..100, RMS and max): circle, mode 7 0.0486 / 0.320 m against
# 0.169 / 0.332 m chasing with mode 3; polyline, mode 7 0.0621 / 0.536 m against 0.104 / 0.702 m.
# Every mode-7 drone ends within 3.1e-6 m of its path's end.  The bounds leave about 25 % (RMS) and
# 20 % (max) above the measured values (DESIGN.md 5f).
BOUNDS = {"circle": (0.06, 0.40), "polyline": (0.08, 0.65)}


@pytest.mark.parametrize("path", ["circle", "polyline"])
def test_oracle_loop_tracks_paths(oracle_mod, path):
    op = oracle_mod.make_params(horizon=N_LOOP, dt=DT, convergence_tolerance=1e-3)
    P, V = (circle_paths if path == "circle" else polyline_paths)(128, T_PATH, DT)
    p0, v0 = P[:, 0].copy(), V[:, 0].copy()
    p7, _, h7 = track_oracle.closed_loop(op, 7, p0, v0, (P, V), STEPS, record=True)
    h3 = chase_loop(op, p0, v0, P, STEPS)
    rms7, max7 = loop_errors(h7, P)
    rms3, max3 = loop_errors(h3, P)
    print(f"\n{path}: mode 7 rms {rms7:.4g} max {max7:.4g}; mode 3 chasing rms {rms3:.4g} max {max3:.4g}; "
          f"end {np.linalg.norm(p7 - P[:, -1], axis=1).max():.3g}")
    assert rms7 < rms3 and max7 < max3
    b_rms, b_max = BOUNDS[path]
    assert rms7 <= b_rms and max7 <= b_max, (rms7, max7)
    assert np.linalg.norm(p7 - P[:, -1], axis=1).max() <= 1e-4


def test_oracle_loop_tracks_through_the_sphere_world(oracle_mod):
    """Straight paths through the 48-sphere world: mode 7 follows them into the spheres, mode 8 with
    the analytic list (margin 1 m) leaves them where they cross one; collisions judged on the
    rasterised map as in test_sphere_mode."""
    og, p0, goal = sphere_world(oracle_mod)
    from dart_planner_b200.mission import reference_path
    P, V = reference_path(np.stack([p0, goal], 1), 2.0, DT, STEPS)
    op = oracle_mod.make_params(horizon=N_LOOP, dt=DT, convergence_tolerance=1e-3)
    s = world_list()
    counts = {}
    for mode in (7, 8):
        _, _, h = track_oracle.closed_loop(op, mode, p0, V[:, 0], (P, V), STEPS, s if mode == 8 else None, W, 1.0,
                                           record=True)
        prev = np.concatenate([p0[None], h[:-1]])
        hit = np.zeros(len(p0), bool)
        for k in range(STEPS):
            hit |= path_collides(og.occ, ORIGIN, RES, og.g.prior, prev[k], h[k], 0.0, 0.6)
        counts[mode] = int(hit.sum())
    print(f"\nsphere world, {len(p0)} drones: collisions mode 7 {counts[7]}, mode 8 {counts[8]}")
    assert counts[8] < counts[7]
    assert counts == SPHERE_WORLD_COUNTS


# Measured: 26 of 256 drones collide in mode 7, none in mode 8 (margin 1 m, w 1000).
SPHERE_WORLD_COUNTS = {7: 26, 8: 0}
