"""Exact-arithmetic checks of results of the tracking modes 7 and 8, on top of ``exact_check``
and ``sphere_exact`` (the same three checks, with the tracking terms in place of the goal and zero
velocity targets):

(a) ``cost`` is f(x): sum_k wpf_k |P_k - r_k|^2 + w_vel |V_k - u_k|^2 + w_acc |a_k|^2 +
    w_thrust |T_k - m g e3|^2 (+ the sphere sum in mode 8) at the returned rows, over Fractions,
    within 64 eps times the sum of the term magnitudes.
(b) the P/V rows are the exact rollout of the thrusts (``exact_check.rollout_ratio``).
(c) a CONV_PGTOL stop is honest for the adjoint thrust gradient with dP_k = 2 w_pos (P_k - r_k)
    (x 11 at k = N-1) plus the sphere gradient, and dV_k = 2 w_vel (V_k - u_k), at the exact
    rolled-out states.  Formula depth: the mode-3 bound of ``sphere_exact`` plus one rounding for
    each target subtraction.
The targets of one problem are given as rp, rv (N, 3): the samples its timesteps read.
"""
from fractions import Fraction as Fr
import math

import numpy as np

import exact_check as ec
import sphere_exact as se


def window(P, V, start, N):
    """the (N, 3) targets of a solve whose timestep k reads sample min(start + k, T - 1)"""
    j = np.minimum(start + np.arange(N), P.shape[0] - 1)
    return P[j], (np.zeros((N, 3)) if V is None else V[j])


def cost_error(params, rp, rv, pos_on, x, cost, spheres=None, w=0.0, margin=0.0):
    q = ec._P(params)
    N, m, g = q["N"], q["mass"], q["gravity"]
    X = [Fr(float(v)) for v in x]
    xa = np.abs(np.asarray(x, np.float64))
    fm, gm = float(m), float(g)
    f, mag = Fr(0), 0.0
    for k in range(N):
        for c in range(3):
            P, V, T = X[3 * k + c], X[3 * N + 3 * k + c], X[6 * N + 3 * k + c]
            Pa, Va, Ta = xa[3 * k + c], xa[3 * N + 3 * k + c], xa[6 * N + 3 * k + c]
            if pos_on:
                e = P - Fr(float(rp[k][c]))
                wp = q["w_pos"] * (11 if k == N - 1 else 1)
                f += wp * e * e
                mag += float(wp) * (Pa + abs(rp[k][c])) ** 2
            ev = V - Fr(float(rv[k][c]))
            f += q["w_vel"] * ev * ev
            mag += float(q["w_vel"]) * (Va + abs(rv[k][c])) ** 2
            a = T / m - (g if c == 2 else 0)
            f += q["w_acc"] * a * a
            mag += float(q["w_acc"]) * (Ta / fm + (gm if c == 2 else 0.0)) ** 2
            d = T - (q["hover"] if c == 2 else 0)
            f += q["w_thrust"] * d * d
            mag += float(q["w_thrust"]) * (Ta + (fm * gm if c == 2 else 0.0)) ** 2
        if spheres is not None:
            pf, _, pabs, _ = se.penalty(spheres, w, margin, x[3 * k:3 * k + 3])
            f += pf
            mag += pabs
    return float(abs(Fr(float(cost)) - f)) / (ec.COST_FACTOR * ec.EPS * mag)


def projected_gradient_excess(params, p0, v0, rp, rv, pos_on, x, spheres=None, w=0.0, margin=0.0):
    q = ec._P(params)
    N, m, g, hover, dt = q["N"], q["mass"], q["gravity"], q["hover"], q["dt"]
    fm, fg, fdt = float(m), float(g), float(dt)
    S = np.zeros((0, 4)) if spheres is None else np.asarray(spheres, np.float64).reshape(-1, 4)
    T = np.asarray(x[6 * N:], np.float64).reshape(N, 3)
    P, V, Pa, Va = ec.rollout(params, p0, v0, T)
    mu, nu, mua, nua = [Fr(0)] * 3, [Fr(0)] * 3, np.zeros(3), np.zeros(3)
    G, gabs = [Fr(0)] * (9 * N), np.zeros(9 * N)
    for k in range(N - 1, -1, -1):
        gpen, pga = [Fr(0)] * 3, 0.0
        if len(S):
            _, gpen, _, pga = se.penalty(S, w, margin, P[k])
            pga = max(pga, se.penalty(S, w, margin, x[3 * k:3 * k + 3])[3])
        for c in range(3):
            gp, gpa = gpen[c], pga
            if pos_on:
                gp += 2 * q["w_pos"] * (P[k][c] - Fr(float(rp[k][c]))) * (11 if k == N - 1 else 1)
                gpa += 2 * float(q["w_pos"]) * (Pa[k][c] + abs(rp[k][c])) * (11 if k == N - 1 else 1)
            t, ta = Fr(float(T[k][c])), abs(T[k][c])
            gk = 2 * q["w_acc"] * (t / m - (g if c == 2 else 0)) / m + 2 * q["w_thrust"] * (t - (hover if c == 2 else 0))
            gka = (2 * float(q["w_acc"]) * (ta / fm + (fg if c == 2 else 0.0)) / fm
                   + 2 * float(q["w_thrust"]) * (ta + (fm * fg if c == 2 else 0.0)))
            if k < N - 1:
                gk += (dt * dt / 2 * mu[c] + dt * nu[c]) / m
                gka += (fdt * fdt / 2 * mua[c] + fdt * nua[c]) / fm
            G[6 * N + 3 * k + c], gabs[6 * N + 3 * k + c] = gk, gka
            nu[c] = 2 * q["w_vel"] * (V[k][c] - Fr(float(rv[k][c]))) + nu[c] + dt * mu[c]
            nua[c] = 2 * float(q["w_vel"]) * (Va[k][c] + abs(rv[k][c])) + nua[c] + fdt * mua[c]
            mu[c], mua[c] = gp + mu[c], gpa + mua[c]
    K = 16 * N + 42 + len(S)
    lo, hi = ec._bounds(params)
    worst = -math.inf
    for i in range(6 * N, 9 * N):
        gi, xi = G[i], Fr(float(x[i]))
        if gi < 0:
            p, bnd = max(xi - Fr(float(hi[i])), gi), abs(float(hi[i]))
        else:
            p, bnd = min(xi - Fr(float(lo[i])), gi), abs(float(lo[i]))
        allow = ec.gamma(K) * gabs[i] + ec.EPS * (abs(float(x[i])) + bnd)
        worst = max(worst, float(abs(p)) - allow)
    return worst


def check_results(params, p0, v0, ref, start, has_goal, res, sample, spheres=None, w=0.0, margin=0.0, what=""):
    """Checks (a), (b) and (c) on the problems `sample`; ref = (P (B, T, 3), V (B, T, 3) or None).
    Returns the number of CONV_PGTOL stops."""
    N = int(params.horizon)
    n_pg = 0
    for b in sample:
        b = int(b)
        rp, rv = window(ref[0][b], None if ref[1] is None else ref[1][b], start, N)
        pos_on = has_goal is None or bool(has_goal[b])
        x = np.asarray(res.x[b], np.float64)
        if int(res.task[b]) != ec.TASK_ABNORMAL:
            r = cost_error(params, rp, rv, pos_on, x, res.cost[b], spheres, w, margin)
            assert r <= 1.0, f"{what} problem {b}: |cost - f(x)| is {r:.3g} x 64 eps sum|terms|"
        r = ec.rollout_ratio(params, p0[b], v0[b], x)
        assert r <= 1.0, f"{what} problem {b}: P/V rows are not the rollout of the thrusts ({r:.2f} x the bound)"
        if int(res.task[b]) == ec.TASK_PGTOL:
            ex = projected_gradient_excess(params, p0[b], v0[b], rp, rv, pos_on, x, spheres, w, margin)
            assert ex <= float(params.gtol), \
                f"{what} problem {b}: CONV_PGTOL stop with max|proj g| - allowance = {ex:.3e} > gtol {params.gtol}"
            n_pg += 1
    return n_pg
