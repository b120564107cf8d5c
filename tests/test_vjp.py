"""The differentiable solve (dart_se3mpc_solve_vjp_batch), CPU tier: the dense restatement
(tests/vjp_oracle.py) against the mode oracles' objectives and against central differences of tight
oracle solves, the kernel's device routine built for the host (tests/emu_vjp) against the restatement
in all four modes, the indefinite case, and the C ABI's refusals."""
import ctypes as C
import os

import numpy as np
import pytest

import emu_vjp
import rollout_oracle
import sphere_oracle
import track_oracle
import vjp_oracle
from test_rollout_mode import _inputs
from test_sphere_mode import MARGIN, W

DT = 0.1


def _params(mode, N, tol=5e-2, **cfg):
    from dart_planner_b200.config import SE3MPCConfig, make_params
    return make_params(SE3MPCConfig(prediction_horizon=N, dt=DT, convergence_tolerance=tol, obstacle_weight=W, **cfg),
                       gradient_mode=mode)


def _box(p, N):
    return (np.tile([-p.tilt_thrust, -p.tilt_thrust, p.min_thrust], N),
            np.tile([p.tilt_thrust, p.tilt_thrust, p.max_thrust], N))


def _random_case(p, mode, N, B, seed):
    """Starts, goals or references, a sphere list near the starts (modes 6 / 8), and thrusts in the box
    with about a fifth of the entries on a bound."""
    rng = np.random.default_rng(seed)
    p0, v0, goal, hg = _inputs(B, seed)
    r = u = s = None
    if mode in (7, 8):
        r = (p0[:, None] + rng.normal(0, 0.6, (B, N, 3)).cumsum(1)).reshape(B, 3 * N)
        u = rng.normal(0, 2, (B, 3 * N))
    if mode in (6, 8):
        s = np.array([[*(p0[0] + [0.5, 0.0, 0.3]), 1.0], [*(p0[1] - [0.2, 0.4, 0.0]), 1.5], [50.0, 50.0, 50.0, 1.0]])
    lo, hi = _box(p, N)
    T = np.tile([0.0, 0.0, p.mass * p.gravity], N) + rng.normal(0, 6, (B, 3 * N))
    T = np.clip(T, lo, hi)
    return p0, v0, goal, hg, r, u, s, T


def _rel(a, b):
    """max over problems of |a - b| / max|b| (per problem and output)"""
    scale = np.maximum(np.abs(b).max(1), 1e-300)
    return (np.abs(a - b).max(1) / scale).max()


# ---- the restatement's objective is the modes' ------------------------------------------------------
@pytest.mark.parametrize("N", [1, 8, 16])
@pytest.mark.parametrize("mode", [3, 6, 7, 8])
def test_restatement_objective_matches_the_mode_oracles(oracle_mod, mode, N):
    op = oracle_mod.make_params(horizon=N, dt=DT)
    p0, v0, goal, hg, r, u, s, T = _random_case(op, mode, N, 12, 7 + N)
    pr = vjp_oracle.Problems(op, p0, v0, goal=None if r is not None else goal, r=r, u=u, has_goal=hg, spheres=s,
                             weight=W, margin=MARGIN)
    f, g = pr.fg(T)
    for b in range(12):
        if mode == 3:
            fo, go = rollout_oracle.dynamics_fg(op, p0[b], v0[b], goal[b] if hg[b] else None, T[b])
        elif mode == 6:
            fo, go = sphere_oracle.fg(op, 6, p0[b], v0[b], goal[b] if hg[b] else None, T[b], s, W, MARGIN)
        else:
            fo, go = track_oracle.fg(op, mode, p0[b], v0[b], (r[b].reshape(N, 3), u[b].reshape(N, 3)), T[b],
                                     s, W, MARGIN, has_goal=bool(hg[b]))
        assert f[b] == pytest.approx(fo, rel=1e-12, abs=0)
        assert np.abs(g[b] - go).max() <= 1e-12 * max(np.abs(go).max(), 1.0)


# ---- the restatement against central differences of tight solves -------------------------------------
def _tight_solve(op, mode, p0, v0, goal, r, u, hg):
    """The oracle's L-BFGS-B at gtol 1e-12, then Newton steps on its free set with the oracle's own
    gradient (the objective is a quadratic in T): the optimum to rounding, with the solve's active set."""
    N = op.horizon
    if mode == 3:
        res = rollout_oracle.solve_batch(op, p0, v0, goal, has_goal=hg)
    else:
        res = track_oracle.solve_batch(op, 7, p0, v0, (r.reshape(-1, N, 3), u.reshape(-1, N, 3)), has_goal=hg)
    T = res.x[:, 6 * N:].copy()
    pr = vjp_oracle.Problems(op, p0, v0, goal=goal if mode == 3 else None, r=r, u=u, has_goal=hg)
    H, _ = pr.hessian(T)
    F = ~pr.active(T)
    for b in range(len(T)):
        for _ in range(2):
            if mode == 3:
                _, g = rollout_oracle.dynamics_fg(op, p0[b], v0[b], goal[b] if hg[b] else None, T[b])
            else:
                _, g = track_oracle.fg(op, 7, p0[b], v0[b], (r[b].reshape(N, 3), u[b].reshape(N, 3)), T[b],
                                       has_goal=bool(hg[b]))
            f = F[b]
            T[b, f] -= np.linalg.solve(H[b][np.ix_(f, f)], g[f])
    x = np.stack([rollout_oracle.rollout(op, p0[b], v0[b], T[b]) for b in range(len(T))])
    return x, pr.fg(T)[0], pr.active(T)


def _fd_cases(N):
    """interior, saturated (far goals: T_z at max_thrust, lateral thrust at tilt_thrust) and goal-less"""
    rng = np.random.default_rng(N)
    p0 = rng.uniform(-3, 3, (6, 3))
    v0 = rng.uniform(-0.3, 0.3, (6, 3))
    goal = p0 + rng.uniform(-0.5, 0.5, (6, 3))
    goal[2:4] = p0[2:4] + [[60.0, -45.0, 90.0], [-70.0, 30.0, 120.0]]
    hg = np.ones(6, np.uint8)
    hg[4] = 0
    return p0, v0, goal, hg


@pytest.mark.parametrize("N", [1, 8, 16])
@pytest.mark.parametrize("mode", [3, 7])
def test_restatement_matches_central_differences(oracle_mod, mode, N):
    op = oracle_mod.make_params(horizon=N, dt=DT, convergence_tolerance=1e-12, max_iterations=5000)
    p0, v0, goal, hg = _fd_cases(N)
    r = u = None
    if mode == 7:
        rng = np.random.default_rng(100 + N)
        r = (goal[:, None] + rng.normal(0, 0.1, (6, N, 3))).reshape(6, 3 * N)
        r[2:4] = (p0[2:4, None] + np.array([60.0, -45.0, 90.0]) * np.linspace(0.2, 1, N)[None, :, None]).reshape(2, -1)
        u = rng.normal(0, 0.3, (6, 3 * N))
    x, cost, act = _tight_solve(op, mode, p0, v0, goal, r, u, hg)
    pr = vjp_oracle.Problems(op, p0, v0, goal=goal if mode == 3 else None, r=r, u=u, has_goal=hg)
    dx, dc, status = pr.plan_jacobian(x[:, 6 * N:])
    assert (status == 0).all()
    assert not act[:2].any()                                   # interior
    assert N == 1 or act[2:4].sum() >= 2 * N                   # saturated (at N = 1, T_0 enters no state)
    names = ["w_pos", "w_vel", "w_acc", "w_thrust"]
    K = pr.theta_size()
    for j in range(K):
        def solve(sign):
            q = oracle_mod.make_params(horizon=N, dt=DT, convergence_tolerance=1e-12, max_iterations=5000)
            pp, vv, gg = p0.copy(), v0.copy(), goal.copy()
            rr, uu = (None, None) if r is None else (r.copy(), u.copy())
            if j >= K - 4:
                h = 1e-4 * getattr(q, names[j - K + 4])
                setattr(q, names[j - K + 4], getattr(q, names[j - K + 4]) + sign * h)
            else:
                h = 1e-3
                if j < 3:
                    pp[:, j] += sign * h
                elif j < 6:
                    vv[:, j - 3] += sign * h
                elif mode == 3:
                    gg[:, j - 6] += sign * h
                elif j < 6 + 3 * N:
                    rr[:, j - 6] += sign * h
                else:
                    uu[:, j - 6 - 3 * N] += sign * h
            return _tight_solve(q, mode, pp, vv, gg, rr, uu, hg), h
        (xp, cp, ap), h = solve(1)
        (xm, cm, am), _ = solve(-1)
        assert (ap == act).all() and (am == act).all(), j       # the perturbation keeps the active set
        fx, fc = (xp - xm) / (2 * h), (cp - cm) / (2 * h)
        # 1e-6 relative, beside the rounding of the differenced values themselves
        sx = np.maximum(np.abs(dx[:, :, j]).max(1), 1e-3)
        assert (np.abs(fx - dx[:, :, j]).max(1) / sx).max() <= 1e-6, j
        tol = 1e-6 * np.maximum(np.abs(dc[:, j]), 1e-3) + 8 * 2.2e-16 * np.abs(cost) / h
        assert (np.abs(fc - dc[:, j]) <= tol).all(), (j, np.abs(fc - dc[:, j]), tol)


# ---- the device routine (host build) against the restatement ------------------------------------------
@pytest.mark.parametrize("N", [1, 4, 8, 13, 16])
@pytest.mark.parametrize("mode", [3, 6, 7, 8])
def test_core_matches_restatement(mode, N):
    p = _params(mode, N)
    B = 48
    p0, v0, goal, hg, r, u, s, T = _random_case(p, mode, N, B, 31 * N + mode)
    rng = np.random.default_rng(N)
    x = np.zeros((B, 9 * N))
    x[:, 6 * N:] = T
    x[:, :6 * N] = rng.normal(size=(B, 6 * N))                  # not read
    gx, gc = rng.normal(size=(B, 9 * N)), rng.normal(size=B)
    gx[::5], gc[1::5] = 0.0, 0.0                                  # one of the two upstream gradients alone
    pr = vjp_oracle.Problems(p, p0, v0, goal=None if r is not None else goal, r=r, u=u, has_goal=hg, spheres=s,
                             weight=W, margin=MARGIN)
    want = pr.vjp(T, gx, gc)
    ref = None if r is None else np.concatenate([r, u], 1)
    got = emu_vjp.vjp_batch(p, p0, v0, goal, x, gx, gc, ref=ref, spheres=s, margin=MARGIN, has_goal=hg)
    assert (got["status"] == want["status"]).all()
    ok = want["status"] == 0
    assert ok.mean() > 0.9
    for k in ("gp0", "gv0", "gw", "gref" if r is not None else "ggoal"):
        assert _rel(got[k][ok], want[k][ok]) <= 1e-10, k
        assert np.isnan(got[k][~ok]).all(), k


def test_core_at_oracle_solutions(oracle_mod):
    """At the points the solve returns (converged or stopped by its iteration limit)."""
    N = 8
    op = oracle_mod.make_params(horizon=N, dt=DT)
    p = _params(3, N)
    p0, v0, goal, hg = _inputs(64, 5)
    x = rollout_oracle.solve_batch(op, p0, v0, goal, has_goal=hg).x
    rng = np.random.default_rng(1)
    gx, gc = rng.normal(size=(64, 9 * N)), rng.normal(size=64)
    want = vjp_oracle.Problems(p, p0, v0, goal, has_goal=hg).vjp(x[:, 6 * N:], gx, gc)
    got = emu_vjp.vjp_batch(p, p0, v0, goal, x, gx, gc, has_goal=hg)
    assert (got["status"] == 0).all() and (want["status"] == 0).all()
    for k in ("gp0", "gv0", "ggoal", "gw"):
        assert _rel(got[k], want[k]) <= 1e-10, k


def test_indefinite_case_gives_status_1_and_nan():
    """Mode 6: a position deep inside a sphere makes H_FF indefinite."""
    N = 8
    p = _params(6, N)
    p0 = np.array([[0.0, 0.0, 5.0], [20.0, 0.0, 5.0]])
    v0 = np.zeros((2, 3))
    goal = p0 + [3.0, 0.0, 0.0]
    s = np.array([[0.0, 0.0, 5.0, 3.0]])                          # centred on the first start
    T = np.tile([0.0, 0.0, p.mass * p.gravity], (2, N))
    x = np.zeros((2, 9 * N))
    x[:, 6 * N:] = T
    gx = np.ones((2, 9 * N))
    want = vjp_oracle.Problems(p, p0, v0, goal, spheres=s, weight=W, margin=MARGIN).vjp(T, gx)
    got = emu_vjp.vjp_batch(p, p0, v0, goal, x, gx, None, spheres=s, margin=MARGIN)
    assert list(want["status"]) == [1, 0] and list(got["status"]) == [1, 0]
    for k in ("gp0", "gv0", "ggoal", "gw"):
        assert np.isnan(got[k][0]).all() and np.isfinite(got[k][1]).all()
        assert _rel(got[k][1:], want[k][1:]) <= 1e-10
    # status 1 belongs to the system solved, H_FF lam_F = tbar_F: without upstream gradients tbar_F = 0,
    # lam = 0 solves it, and both give status 0 and zero gradients
    want = vjp_oracle.Problems(p, p0, v0, goal, spheres=s, weight=W, margin=MARGIN).vjp(T)
    got = emu_vjp.vjp_batch(p, p0, v0, goal, x, None, None, spheres=s, margin=MARGIN)
    assert list(want["status"]) == [0, 0] and list(got["status"]) == [0, 0]
    for k in ("gp0", "gv0", "ggoal", "gw"):
        assert (got[k] == 0).all() and (want[k] == 0).all()


def _contact_case(op, mode, N, seed):
    """Thrusts, starts and targets with spheres around positions of a few timesteps and one out of reach:
    the penalty's Hessian enters H and dg/dtheta.  No position within 1e-2 of a surface (h = 0), where the
    penalty is only once differentiable: the first seed from `seed` on that gives such a case."""
    while True:
        rng = np.random.default_rng(seed)
        B = 4
        p0, v0 = rng.uniform(-3, 3, (B, 3)), rng.uniform(-1, 1, (B, 3))
        goal = p0 + rng.uniform(-2, 2, (B, 3))
        T = np.tile([0.0, 0.0, op.mass * op.gravity], N) + rng.normal(0, 2, (B, 3 * N))
        r = u = None
        if mode == 8:
            r = (goal[:, None] + rng.normal(0, 0.5, (B, N, 3))).reshape(B, 3 * N)
            u = rng.normal(0, 1, (B, 3 * N))
        P, _, _ = vjp_oracle.Problems(op, p0, v0, goal).states(T)
        P = P.reshape(B, N, 3)
        s = np.array([[*(P[0, N - 1] + [0.3, -0.2, 0.1]), 1.2], [*(P[1, N // 2] - [0.1, 0.4, 0.0]), 1.0],
                      [*(P[2, 1] + [0.0, 0.0, 0.5]), 1.1], [60.0, 60.0, 60.0, 1.0]])
        e = P[:, :, None] - s[None, None, :, :3]
        hh = (s[None, None, :, 3] + MARGIN) ** 2 - (e * e).sum(-1)
        if (np.abs(hh) > 1e-2).all():
            assert (hh > 0).sum() >= 3
            return p0, v0, goal, r, u, T, s
        seed += 1000


@pytest.mark.parametrize("N", [2, 8, 16])
@pytest.mark.parametrize("mode", [6, 8])
def test_restatement_second_derivatives_match_differences_of_its_gradient(oracle_mod, mode, N):
    """With spheres the restatement's H (8 w e e^T - 4 w h I on the contacts) and dg/dtheta against central
    differences of its own g, whose agreement with the mode oracles is tested above; df/dtheta against
    differences of f."""
    names = ["position_weight", "velocity_weight", "acceleration_weight", "thrust_weight"]
    base = dict(position_weight=100.0, velocity_weight=10.0, acceleration_weight=1.0, thrust_weight=0.1)
    op = oracle_mod.make_params(horizon=N, dt=DT)
    p0, v0, goal, r, u, T, s = _contact_case(op, mode, N, N + mode)

    def problems(op=op, p0=p0, v0=v0, goal=goal, r=r, u=u):
        return vjp_oracle.Problems(op, p0, v0, goal=None if r is not None else goal, r=r, u=u, spheres=s, weight=W,
                                   margin=MARGIN)

    pr = problems()
    H, _ = pr.hessian(T)
    G, df, _ = pr.jacobians(T)
    f0, g0 = pr.fg(T)
    h = 1e-5
    num = np.stack([(pr.fg(T + h * d)[1] - pr.fg(T - h * d)[1]) / (2 * h) for d in np.eye(3 * N)], 2)
    assert np.abs(num - H).max() <= 1e-6 * np.abs(H).max()
    K = pr.theta_size()
    for j in range(K):
        def at(sign):
            if j >= K - 4:
                w = dict(base)
                hj = 1e-6 * w[names[j - K + 4]]
                w[names[j - K + 4]] += sign * hj
                return problems(op=oracle_mod.make_params(horizon=N, dt=DT, **w)), hj
            hj, a = 1e-5, [p0.copy(), v0.copy(), goal.copy(), None if r is None else r.copy(),
                           None if u is None else u.copy()]
            if j < 6:
                a[j // 3][:, j % 3] += sign * hj
            elif mode == 6:
                a[2][:, j - 6] += sign * hj
            elif j < 6 + 3 * N:
                a[3][:, j - 6] += sign * hj
            else:
                a[4][:, j - 6 - 3 * N] += sign * hj
            return problems(p0=a[0], v0=a[1], goal=a[2], r=a[3], u=a[4]), hj
        (pp, hj), (pm, _) = at(1), at(-1)
        (fp, gp), (fm, gm) = pp.fg(T), pm.fg(T)
        assert np.abs((gp - gm) / (2 * hj) - G[:, :, j]).max() <= 1e-6 * max(np.abs(G).max(), 1.0), j
        assert (np.abs((fp - fm) / (2 * hj) - df[:, j]) <= 1e-6 * np.abs(df).max() + 1e-15 * np.abs(f0) / hj).all(), j


# ---- the C ABI's refusals (no GPU needed: they come before any CUDA call) -------------------------------
def vjp_call(L, q, B=0, ld=None, x=True, status=True, goal=True, ref=None, sph=None, buf=None):
    bp = buf.ctypes.data
    return L.dart_se3mpc_solve_vjp_batch(C.byref(q), B, B if ld is None else ld, bp, bp, bp if goal else None, None,
                                         bp if x else None, None if ref is None else C.byref(ref),
                                         None if sph is None else C.byref(sph), None, None, None, None, None, None,
                                         None, bp if status else None, None)


def check_refusals(L):
    from dart_planner_b200 import _cabi
    OK, BAD, UNS = _cabi.DART_OK, _cabi.DART_E_BADARG, _cabi.DART_E_UNSUPPORTED
    buf = np.zeros(64 * 9 * 16)
    lst = np.zeros((2, 4))
    sph = _cabi.Spheres(2, 0, lst.ctypes.data, 0.5)

    def ref(N=8, start=0, rows=True):
        return _cabi.TrackRef(N, start, buf.ctypes.data if rows else None)

    def q(mode, N=8):
        p = _params(0, N)
        p.gradient_mode = mode
        return p

    def call(p, **kw):
        return vjp_call(L, p, buf=buf, **kw)

    assert call(q(3)) == OK and call(q(6), sph=sph) == OK
    assert call(q(7), ref=ref()) == OK and call(q(8), ref=ref(), sph=sph) == OK
    assert call(q(8), ref=ref(), sph=_cabi.Spheres(0, 0, None, 0.5)) == OK       # an empty list
    for mode in (0, 1, 2, 4, 5, 9, -1):
        assert call(q(mode)) == BAD and call(q(mode), sph=sph) == BAD and call(q(mode), ref=ref()) == BAD, mode
    assert call(q(3), sph=sph) == BAD and call(q(7), ref=ref(), sph=sph) == BAD   # spheres in 3 / 7
    assert call(q(6)) == BAD and call(q(8), ref=ref()) == BAD                     # none in 6 / 8
    assert call(q(6), sph=_cabi.Spheres(-1, 0, lst.ctypes.data, 0.5)) == BAD
    assert call(q(6), sph=_cabi.Spheres(1, 0, None, 0.5)) == BAD
    assert call(q(3), ref=ref()) == BAD and call(q(6), ref=ref(), sph=sph) == BAD # a reference in 3 / 6
    assert call(q(7)) == BAD and call(q(8), sph=sph) == BAD                       # none in 7 / 8
    assert call(q(7), ref=ref(N=9)) == BAD and call(q(7), ref=ref(start=1)) == BAD
    assert call(q(7), ref=ref(rows=False)) == BAD
    assert call(q(3), x=False) == BAD and call(q(3), status=False) == BAD and call(q(3), goal=False) == BAD
    assert call(q(7), ref=ref(), goal=False) == OK                                # no goal in 7 / 8
    assert call(q(3), B=4, ld=2) == BAD
    assert call(q(3, 17)) == UNS and call(q(7, 17), ref=ref(N=17)) == UNS and call(q(3, 16)) == OK
    assert call(q(6, 17), sph=sph) == UNS and call(q(8, 1), ref=ref(N=1), sph=sph) == OK


def test_vjp_entry_refuses_bad_arguments_without_a_gpu():
    from dart_planner_b200 import _cabi
    if not os.path.exists(_cabi.LIB_PATH):
        pytest.skip("library not built")
    check_refusals(_cabi.lib())
