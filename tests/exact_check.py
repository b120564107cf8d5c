"""Exact-arithmetic checks of solver results, independent of the oracle and of the kernel.

Everything is evaluated with `fractions.Fraction` on the float values a solver returned, so the
only rounding left is the solver's own.  Three checks, for every gradient mode:

(a) ``cost`` is f(x): the reference objective (orc_objective, se3_mpc_planner.py:516-550) plus, in
    modes 2 and 4, the occupancy penalty sum_k w max(0, o(P_k) - free_level)^2.  o is written as the
    explicit sum over the eight corners of the trilinear product weights (not the nested lerps of
    the kernel and the oracle); cells are read as stored (float32 or float64), the prior outside the
    grid.  Bound: |cost - f| <= 64 eps sum|terms|, where sum|terms| is f evaluated with every
    operand replaced by its magnitude (a - b -> |a| + |b|).
(b) modes 3 and 4: the P/V rows are the exact rollout of the thrusts, a = T/m - g e3,
    p += v dt + a dt^2/2, v += a dt, to gamma(8(k+1)) times the magnitude of the entry (k its step).
(c) a CONV_PGTOL stop (task 1) is honest: the gradient the mode defines (mode 0 the reference's
    formula, mode 1 the true gradient of f, mode 2 the reference's formula plus the penalty
    gradient, modes 3/4 the thrust gradient of the rolled-out objective), projected on the bounds of
    orc_bounds (oracle/se3mpc_oracle.c:74-91; in modes 3/4 only the thrusts are variables), has
    max |proj g| <= gtol up to the rounding allowance below.

The rounding allowance of (c), derived rather than tuned: the solver computed its projected
gradient p_i in floating point and stopped because max |p_i| <= gtol.  The projection
(min(x - l, g) or max(x - u, g)) is 1-Lipschitz in g and x - l is one rounding, so
|p_i - p_exact_i| <= |g_i - g_exact_i| + eps |x_i - bound_i|.  With the standard forward-error
bound of a formula of depth K (K successive roundings on the longest path, gamma_K =
K eps / (1 - K eps)), |g_i - g_exact_i| <= gamma_K gabs_i, gabs the gradient evaluated with every
operand replaced by its magnitude.  The depths: mode 0: 4 (difference, product, scaling); mode 1:
12 (quotients, differences, products, the terminal sum); mode 2: 24 (mode 0 plus u = p/res - 1/2,
the weights, the corner sums, rho, the product); modes 3/4: 16N + 32 (8 roundings per step of the
rollout that feeds P and V, 4 per step of the adjoint sums, the direct terms and the penalty).
The penalty's magnitudes bound every interpolation weight by 1, so any intermediate of o is at most
sum|c| over the eight corners and any difference quotient at most 2 sum|c| / res.

The cell and the weight t come from u = p/res - 1/2 formed in IEEE double, as the definition
states and as both solvers form it; on a voxel-centre plane o is continuous, its gradient is
one-sided, and the side is the one the rounded u selects.  The kernel's t = u - floor(u) is itself
one more rounding of at most eps, inside the magnitudes above.
"""
from fractions import Fraction as Fr
import math

import numpy as np

EPS = float(np.finfo(np.float64).eps)
COST_FACTOR = 64
TASK_PGTOL, TASK_ABNORMAL = 1, 5


def gamma(k):
    return k * EPS / (1.0 - k * EPS)


class Grid:
    """The penalty grid as the solvers read it: cells (nz, ny, nx) float32 or float64, voxel key of
    cell (0, 0, 0) = origin_voxel, voxel centres at (key + 1/2) res, prior outside."""

    def __init__(self, occ, origin_voxel, resolution, prior):
        self.occ = np.asarray(occ)
        assert self.occ.dtype in (np.float32, np.float64)
        self.origin = tuple(int(o) for o in origin_voxel)
        self.resolution = float(resolution)
        self.prior = float(prior)

    def cell(self, key):
        i = [key[c] - self.origin[c] for c in range(3)]
        nz, ny, nx = self.occ.shape
        if not (0 <= i[0] < nx and 0 <= i[1] < ny and 0 <= i[2] < nz):
            return self.prior
        return float(self.occ[i[2], i[1], i[0]])


def penalty(grid, w, free_level, p):
    """Exact (f, grad[3]) of w max(0, o(p) - free_level)^2 and the magnitudes (fabs, gabs)."""
    res = Fr(grid.resolution)
    key, t = [], []
    for c in range(3):
        u_fp = float(p[c]) / grid.resolution - 0.5           # IEEE double: selects the cell
        k = math.floor(u_fp)
        key.append(k)
        t.append(Fr(u_fp) - k)
    o, do = Fr(0), [Fr(0)] * 3
    cabs = 0.0
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                cv = grid.cell((key[0] + dx, key[1] + dy, key[2] + dz))
                cabs += abs(cv)
                c = Fr(cv)
                wx = t[0] if dx else 1 - t[0]
                wy = t[1] if dy else 1 - t[1]
                wz = t[2] if dz else 1 - t[2]
                o += wx * wy * wz * c
                do[0] += (1 if dx else -1) * wy * wz * c
                do[1] += (1 if dy else -1) * wx * wz * c
                do[2] += (1 if dz else -1) * wx * wy * c
    rho_abs = cabs + abs(free_level)
    fabs = w * rho_abs * rho_abs
    gabs = 2 * w * rho_abs * 2 * cabs / grid.resolution
    rho = o - Fr(free_level)
    if rho <= 0:
        return Fr(0), [Fr(0)] * 3, fabs, gabs
    W = Fr(w)
    return W * rho * rho, [2 * W * rho * d / res for d in do], fabs, gabs


def _P(params):
    q = {k: Fr(float(getattr(params, k))) for k in ("dt", "mass", "gravity", "w_pos", "w_vel", "w_acc", "w_thrust")}
    q["N"] = int(params.horizon)
    q["hover"] = q["mass"] * q["gravity"]
    return q


def objective(params, x, goal, grid=None, w_obs=0.0, free_level=0.5):
    """Exact f(x) (+ penalty with a grid) and sum|terms|."""
    q = _P(params)
    N, m, g = q["N"], q["mass"], q["gravity"]
    X = [Fr(float(v)) for v in x]
    xa = np.abs(np.asarray(x, np.float64))
    fm, gm = float(m), float(g)
    f, mag = Fr(0), 0.0
    for k in range(N):
        for c in range(3):
            P, V, T = X[3 * k + c], X[3 * N + 3 * k + c], X[6 * N + 3 * k + c]
            Pa, Va, Ta = xa[3 * k + c], xa[3 * N + 3 * k + c], xa[6 * N + 3 * k + c]
            if goal is not None:
                e = P - Fr(float(goal[c]))
                wp = q["w_pos"] * (11 if k == N - 1 else 1)
                f += wp * e * e
                mag += float(wp) * (Pa + abs(goal[c])) ** 2
            f += q["w_vel"] * V * V
            mag += float(q["w_vel"]) * Va * Va
            a = T / m - (g if c == 2 else 0)
            f += q["w_acc"] * a * a
            mag += float(q["w_acc"]) * (Ta / fm + (gm if c == 2 else 0.0)) ** 2
            d = T - (q["hover"] if c == 2 else 0)
            f += q["w_thrust"] * d * d
            mag += float(q["w_thrust"]) * (Ta + (fm * gm if c == 2 else 0.0)) ** 2
        if grid is not None:
            pf, _, pabs, _ = penalty(grid, w_obs, free_level, x[3 * k:3 * k + 3])
            f += pf
            mag += pabs
    return f, mag


def rollout(params, p0, v0, T):
    """Exact P, V (lists of N x 3 Fractions) of the plant from (p0, v0) under thrusts T (N, 3),
    and their magnitudes (the same recursion on |.|)."""
    q = _P(params)
    N, dt, m, g = q["N"], q["dt"], q["mass"], q["gravity"]
    fdt, fm, fg = float(dt), float(m), float(g)
    P = [[Fr(float(p0[c])) for c in range(3)]]
    V = [[Fr(float(v0[c])) for c in range(3)]]
    Pa = [np.abs(np.asarray(p0, np.float64))]
    Va = [np.abs(np.asarray(v0, np.float64))]
    for k in range(N - 1):
        a = [Fr(float(T[k][c])) / m - (g if c == 2 else 0) for c in range(3)]
        aa = np.abs(np.asarray(T[k], np.float64)) / fm + np.array([0.0, 0.0, fg])
        P.append([P[k][c] + V[k][c] * dt + a[c] * dt * dt / 2 for c in range(3)])
        V.append([V[k][c] + a[c] * dt for c in range(3)])
        Pa.append(Pa[k] + Va[k] * fdt + 0.5 * aa * fdt * fdt)
        Va.append(Va[k] + aa * fdt)
    return P, V, np.array(Pa), np.array(Va)


def rollout_ratio(params, p0, v0, x):
    """max over the P/V entries of |x - exact rollout| / (gamma(8(k+1)) magnitude): <= 1 passes."""
    N = int(params.horizon)
    T = np.asarray(x[6 * N:], np.float64).reshape(N, 3)
    P, V, Pa, Va = rollout(params, p0, v0, T)
    worst = 0.0
    for k in range(N):
        tol = gamma(8 * (k + 1))
        for c in range(3):
            for got, ex, mag in ((x[3 * k + c], P[k][c], Pa[k][c]), (x[3 * N + 3 * k + c], V[k][c], Va[k][c])):
                err = abs(Fr(float(got)) - ex)
                if err:
                    worst = max(worst, float(err) / (tol * max(mag, 1e-300)))
    return worst


def _bounds(params):
    N = int(params.horizon)
    lo = np.r_[np.full(3 * N, -params.pos_bound), np.full(3 * N, -params.max_velocity),
               np.tile([-params.tilt_thrust, -params.tilt_thrust, params.min_thrust], N)]
    hi = np.r_[np.full(3 * N, params.pos_bound), np.full(3 * N, params.max_velocity),
               np.tile([params.tilt_thrust, params.tilt_thrust, params.max_thrust], N)]
    return lo, hi


def gradient(params, mode, p0, v0, goal, x, grid=None, w_obs=0.0, free_level=0.5):
    """(indices of the variables, exact gradient, magnitudes gabs, formula depth K)."""
    q = _P(params)
    N, m, g, hover = q["N"], q["mass"], q["gravity"], q["hover"]
    fm, fg = float(m), float(g)
    xa = np.abs(np.asarray(x, np.float64))
    X = [Fr(float(v)) for v in x]
    G = [Fr(0)] * (9 * N)
    gabs = np.zeros(9 * N)
    if mode in (0, 1, 2):
        for i in range(3 * N):
            k, c = divmod(i, 3)
            if goal is not None:
                G[i] = 2 * q["w_pos"] * (X[i] - Fr(float(goal[c])))
                gabs[i] = 2 * float(q["w_pos"]) * (xa[i] + abs(goal[c]))
                if mode == 1 and k == N - 1:
                    G[i] += 20 * q["w_pos"] * (X[i] - Fr(float(goal[c])))
                    gabs[i] *= 11
            G[3 * N + i] = 2 * q["w_vel"] * X[3 * N + i]
            gabs[3 * N + i] = 2 * float(q["w_vel"]) * xa[3 * N + i]
            t = X[6 * N + i]
            if mode == 1:
                G[6 * N + i] = (2 * q["w_acc"] * (t / m - (g if c == 2 else 0)) / m
                                + 2 * q["w_thrust"] * (t - (hover if c == 2 else 0)))
                gabs[6 * N + i] = (2 * float(q["w_acc"]) * (xa[6 * N + i] / fm + (fg if c == 2 else 0.0)) / fm
                                   + 2 * float(q["w_thrust"]) * (xa[6 * N + i] + (fm * fg if c == 2 else 0.0)))
            else:
                G[6 * N + i] = 2 * q["w_thrust"] * t
                gabs[6 * N + i] = 2 * float(q["w_thrust"]) * xa[6 * N + i]
        if mode == 2:
            for k in range(N):
                _, gp, _, pga = penalty(grid, w_obs, free_level, x[3 * k:3 * k + 3])
                for c in range(3):
                    G[3 * k + c] += gp[c]
                    gabs[3 * k + c] += pga
        return np.arange(9 * N), G, gabs, {0: 4, 1: 12, 2: 24}[mode]
    # modes 3/4: the thrust gradient of the rolled-out objective (sequential adjoint, exact)
    dt = q["dt"]
    fdt = float(dt)
    T = np.asarray(x[6 * N:], np.float64).reshape(N, 3)
    P, V, Pa, Va = rollout(params, p0, v0, T)
    mu, nu = [Fr(0)] * 3, [Fr(0)] * 3
    mua, nua = np.zeros(3), np.zeros(3)
    GT, GTa = [None] * (3 * N), np.zeros(3 * N)
    for k in range(N - 1, -1, -1):
        if mode == 4:
            Pk = x[3 * k:3 * k + 3]                       # the returned row: the solver's cell choice
            _, _, _, pga = penalty(grid, w_obs, free_level, Pk)
            gpen = _penalty_grad_exact(grid, w_obs, free_level, P[k], Pk)
        for c in range(3):
            gp, gpa = Fr(0), 0.0
            if goal is not None:
                e = P[k][c] - Fr(float(goal[c]))
                gp = 2 * q["w_pos"] * e * (11 if k == N - 1 else 1)
                gpa = 2 * float(q["w_pos"]) * (Pa[k][c] + abs(goal[c])) * (11 if k == N - 1 else 1)
            if mode == 4:
                gp += gpen[c]
                gpa += pga
            t, ta = Fr(float(T[k][c])), abs(T[k][c])
            gk = (2 * q["w_acc"] * (t / m - (g if c == 2 else 0)) / m
                  + 2 * q["w_thrust"] * (t - (hover if c == 2 else 0)))
            gka = (2 * float(q["w_acc"]) * (ta / fm + (fg if c == 2 else 0.0)) / fm
                   + 2 * float(q["w_thrust"]) * (ta + (fm * fg if c == 2 else 0.0)))
            if k < N - 1:
                gk += (dt * dt / 2 * mu[c] + dt * nu[c]) / m
                gka += (fdt * fdt / 2 * mua[c] + fdt * nua[c]) / fm
            GT[3 * k + c], GTa[3 * k + c] = gk, gka
            nu[c] = 2 * q["w_vel"] * V[k][c] + nu[c] + dt * mu[c]
            nua[c] = 2 * float(q["w_vel"]) * Va[k][c] + nua[c] + fdt * mua[c]
            mu[c] = gp + mu[c]
            mua[c] = gpa + mua[c]
    G[6 * N:] = GT
    gabs[6 * N:] = GTa
    return np.arange(6 * N, 9 * N), G, gabs, 16 * N + 32


def _penalty_grad_exact(grid, w, free_level, Pk_exact, Pk_float):
    """Penalty gradient at the exact rolled-out position, in the cell the rounded position selects."""
    res = Fr(grid.resolution)
    key = [math.floor(float(Pk_float[c]) / grid.resolution - 0.5) for c in range(3)]
    t = [Pk_exact[c] / res - Fr(1, 2) - key[c] for c in range(3)]
    o, do = Fr(0), [Fr(0)] * 3
    for dz in (0, 1):
        for dy in (0, 1):
            for dx in (0, 1):
                c = Fr(grid.cell((key[0] + dx, key[1] + dy, key[2] + dz)))
                wx, wy, wz = (t[0] if dx else 1 - t[0]), (t[1] if dy else 1 - t[1]), (t[2] if dz else 1 - t[2])
                o += wx * wy * wz * c
                do[0] += (1 if dx else -1) * wy * wz * c
                do[1] += (1 if dy else -1) * wx * wz * c
                do[2] += (1 if dz else -1) * wx * wy * c
    rho = o - Fr(free_level)
    if rho <= 0:
        return [Fr(0)] * 3
    return [2 * Fr(w) * rho * d / res for d in do]


def projected_gradient_excess(params, mode, p0, v0, goal, x, grid=None, w_obs=0.0, free_level=0.5):
    """max_i (|proj g_i| - allowance_i) over the variables: a CONV_PGTOL stop needs <= gtol."""
    idx, G, gabs, K = gradient(params, mode, p0, v0, goal, x, grid, w_obs, free_level)
    lo, hi = _bounds(params)
    worst = -math.inf
    for i in idx:
        gi, xi = G[i], Fr(float(x[i]))
        if gi < 0:
            p = max(xi - Fr(float(hi[i])), gi)
            bnd = abs(float(hi[i]))
        else:
            p = min(xi - Fr(float(lo[i])), gi)
            bnd = abs(float(lo[i]))
        allow = gamma(K) * gabs[i] + EPS * (abs(float(x[i])) + bnd)
        worst = max(worst, float(abs(p)) - allow)
    return worst


def cost_error(params, mode, goal, x, cost, grid=None, w_obs=0.0, free_level=0.5):
    """|cost - f(x)| / (64 eps sum|terms|): <= 1 passes check (a)."""
    f, mag = objective(params, x, goal, grid if mode in (2, 4) else None, w_obs, free_level)
    return float(abs(Fr(float(cost)) - f)) / (COST_FACTOR * EPS * mag)


def check_results(params, mode, p0, v0, goal, has_goal, res, sample, grid=None, w_obs=0.0, free_level=0.5,
                  what=""):
    """Checks (a), (b) and (c) on the problems `sample` of a result (x, cost, task).  Returns the
    number of CONV_PGTOL stops checked."""
    N = int(params.horizon)
    n_pg = 0
    pen = grid if mode in (2, 4) else None
    for b in sample:
        b = int(b)
        gb = goal[b] if has_goal is None or has_goal[b] else None
        x = np.asarray(res.x[b], np.float64)
        if int(res.task[b]) != TASK_ABNORMAL:          # ABNORMAL reports the last evaluated f
            r = cost_error(params, mode, gb, x, res.cost[b], pen, w_obs, free_level)
            assert r <= 1.0, f"{what} problem {b}: |cost - f(x)| is {r:.3g} x 64 eps sum|terms|"
        if mode >= 3:
            r = rollout_ratio(params, p0[b], v0[b], x)
            assert r <= 1.0, f"{what} problem {b}: P/V rows are not the rollout of the thrusts ({r:.2f} x the bound)"
        if int(res.task[b]) == TASK_PGTOL:
            ex = projected_gradient_excess(params, mode, p0[b], v0[b], gb, x, pen, w_obs, free_level)
            assert ex <= float(params.gtol), \
                f"{what} problem {b}: CONV_PGTOL stop with max|proj g| - allowance = {ex:.3e} > gtol {params.gtol}"
            n_pg += 1
    return n_pg
