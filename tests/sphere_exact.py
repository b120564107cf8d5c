"""Exact-arithmetic checks of results of the sphere-penalty modes 5 and 6, on top of
``exact_check`` (the same three checks, with the sphere sum added where the mode adds it):

(a) ``cost`` is f(x): the reference objective plus sum_k sum_j w max(0, R_j^2 - |P_k - c_j|^2)^2 with
    R_j = r_j + margin, P_k the returned position rows, over Fractions.  Bound: 64 eps times the sum
    of the term magnitudes, the penalty's being w (R^2 + |P|^2-like magnitudes)^2 of the spheres that
    are active or within rounding of it.
(b) mode 6: the P/V rows are the exact rollout of the thrusts (``exact_check.rollout_ratio``).
(c) a CONV_PGTOL stop is honest for the gradient the mode defines: mode 0's formula plus the sphere
    gradient (mode 5), the adjoint thrust gradient with the sphere gradient at the exact rolled-out
    positions entering dP (mode 6).  Formula depth: the base mode's plus 8 roundings of the term
    (e, the products and sums of d2, R, R R, h, (-4 w) h, the product with e) plus one per sphere of
    the running sum; magnitudes as in (a).
"""
from fractions import Fraction as Fr
import math

import numpy as np

import exact_check as ec


def _near(h, habs):
    """the spheres a floating-point evaluation may count as active"""
    return h > -ec.gamma(8) * habs


def penalty(spheres, w, margin, P):
    """Exact (f, grad[3]) of the sphere penalty at the position P (floats or Fractions), and the
    magnitudes (fabs, gabs)."""
    W = Fr(w)
    Pf = [v if isinstance(v, Fr) else Fr(float(v)) for v in P]
    Pa = [abs(float(v)) for v in P]
    f, g, fabs, gabs = Fr(0), [Fr(0)] * 3, 0.0, 0.0
    for cx, cy, cz, r in np.asarray(spheres, np.float64).reshape(-1, 4):
        e = [Pf[0] - Fr(cx), Pf[1] - Fr(cy), Pf[2] - Fr(cz)]
        ea = [Pa[0] + abs(cx), Pa[1] + abs(cy), Pa[2] + abs(cz)]
        R = Fr(float(r)) + Fr(float(margin))
        ra = abs(r) + abs(margin)
        h = R * R - (e[0] * e[0] + e[1] * e[1] + e[2] * e[2])
        habs = ra * ra + sum(a * a for a in ea)
        if _near(float(h), habs):
            fabs += w * habs * habs
            gabs += 4 * w * habs * max(ea)
        if h > 0:
            f += W * h * h
            g = [g[c] - 4 * W * h * e[c] for c in range(3)]
    return f, g, fabs, gabs


def cost_error(params, goal, x, cost, spheres, w, margin):
    N = int(params.horizon)
    f, mag = ec.objective(params, x, goal)
    for k in range(N):
        pf, _, pabs, _ = penalty(spheres, w, margin, x[3 * k:3 * k + 3])
        f += pf
        mag += pabs
    return float(abs(Fr(float(cost)) - f)) / (ec.COST_FACTOR * ec.EPS * mag)


def projected_gradient_excess(params, mode, p0, v0, goal, x, spheres, w, margin):
    N = int(params.horizon)
    n = len(np.asarray(spheres).reshape(-1, 4))
    if mode == 5:
        idx, G, gabs, K = ec.gradient(params, 0, p0, v0, goal, x)
        for k in range(N):
            _, gp, _, pga = penalty(spheres, w, margin, x[3 * k:3 * k + 3])
            for c in range(3):
                G[3 * k + c] += gp[c]
                gabs[3 * k + c] += pga
        K += 8 + n
    else:
        idx, G, gabs, K = _rollout_gradient(params, p0, v0, goal, x, spheres, w, margin)
    lo, hi = ec._bounds(params)
    worst = -math.inf
    for i in idx:
        gi, xi = G[i], Fr(float(x[i]))
        if gi < 0:
            p, bnd = max(xi - Fr(float(hi[i])), gi), abs(float(hi[i]))
        else:
            p, bnd = min(xi - Fr(float(lo[i])), gi), abs(float(lo[i]))
        allow = ec.gamma(K) * gabs[i] + ec.EPS * (abs(float(x[i])) + bnd)
        worst = max(worst, float(abs(p)) - allow)
    return worst


def _rollout_gradient(params, p0, v0, goal, x, spheres, w, margin):
    """exact_check.gradient's mode-3 adjoint with the sphere gradient at the exact P_k in dP"""
    q = ec._P(params)
    N, m, g, hover, dt = q["N"], q["mass"], q["gravity"], q["hover"], q["dt"]
    fm, fg, fdt = float(m), float(g), float(dt)
    T = np.asarray(x[6 * N:], np.float64).reshape(N, 3)
    P, V, Pa, Va = ec.rollout(params, p0, v0, T)
    mu, nu, mua, nua = [Fr(0)] * 3, [Fr(0)] * 3, np.zeros(3), np.zeros(3)
    G, gabs = [Fr(0)] * (9 * N), np.zeros(9 * N)
    for k in range(N - 1, -1, -1):
        _, gpen, _, pga = penalty(spheres, w, margin, P[k])
        _, _, _, pga_f = penalty(spheres, w, margin, x[3 * k:3 * k + 3])
        pga = max(pga, pga_f)
        for c in range(3):
            gp, gpa = gpen[c], pga
            if goal is not None:
                gp += 2 * q["w_pos"] * (P[k][c] - Fr(float(goal[c]))) * (11 if k == N - 1 else 1)
                gpa += 2 * float(q["w_pos"]) * (Pa[k][c] + abs(goal[c])) * (11 if k == N - 1 else 1)
            t, ta = Fr(float(T[k][c])), abs(T[k][c])
            gk = 2 * q["w_acc"] * (t / m - (g if c == 2 else 0)) / m + 2 * q["w_thrust"] * (t - (hover if c == 2 else 0))
            gka = (2 * float(q["w_acc"]) * (ta / fm + (fg if c == 2 else 0.0)) / fm
                   + 2 * float(q["w_thrust"]) * (ta + (fm * fg if c == 2 else 0.0)))
            if k < N - 1:
                gk += (dt * dt / 2 * mu[c] + dt * nu[c]) / m
                gka += (fdt * fdt / 2 * mua[c] + fdt * nua[c]) / fm
            G[6 * N + 3 * k + c], gabs[6 * N + 3 * k + c] = gk, gka
            nu[c] = 2 * q["w_vel"] * V[k][c] + nu[c] + dt * mu[c]
            nua[c] = 2 * float(q["w_vel"]) * Va[k][c] + nua[c] + fdt * mua[c]
            mu[c], mua[c] = gp + mu[c], gpa + mua[c]
    return np.arange(6 * N, 9 * N), G, gabs, 16 * N + 40 + len(np.asarray(spheres).reshape(-1, 4))


def check_results(params, mode, p0, v0, goal, has_goal, res, sample, spheres, w, margin, what=""):
    """Checks (a), (b) and (c) on the problems `sample`; returns the number of CONV_PGTOL stops."""
    n_pg = 0
    for b in sample:
        b = int(b)
        gb = goal[b] if has_goal is None or has_goal[b] else None
        x = np.asarray(res.x[b], np.float64)
        if int(res.task[b]) != ec.TASK_ABNORMAL:
            r = cost_error(params, gb, x, res.cost[b], spheres, w, margin)
            assert r <= 1.0, f"{what} problem {b}: |cost - f(x)| is {r:.3g} x 64 eps sum|terms|"
        if mode == 6:
            r = ec.rollout_ratio(params, p0[b], v0[b], x)
            assert r <= 1.0, f"{what} problem {b}: P/V rows are not the rollout of the thrusts ({r:.2f} x the bound)"
        if int(res.task[b]) == ec.TASK_PGTOL:
            ex = projected_gradient_excess(params, mode, p0[b], v0[b], gb, x, spheres, w, margin)
            assert ex <= float(params.gtol), \
                f"{what} problem {b}: CONV_PGTOL stop with max|proj g| - allowance = {ex:.3e} > gtol {params.gtol}"
            n_pg += 1
    return n_pg
