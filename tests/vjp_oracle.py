"""Dense restatement of the differentiable solve (dart_se3mpc_solve_vjp_batch) -- TEST INFRASTRUCTURE.

It builds the rollout matrices, the Hessian H, the parameter Jacobian dg/dtheta and the direct
derivatives explicitly (batched NumPy), solves H_FF dT_F = -dg_F/dtheta for the whole Jacobian of the
plan, and contracts it with the upstream gradients -- none of the kernel's recursions, scans or
conjugate gradients.  Objective of gradient modes 3, 6, 7 and 8 (include/dart_se3mpc.h):
  f = sum_k wpf_k |P_k - r_k|^2 + w_vel |V_k - u_k|^2 + w_acc |a_k|^2 + w_thrust |T_k - m g e3|^2
      + the sphere penalty on P_k (modes 6 / 8),
with r_k = goal and u_k = 0 in the goal modes, wpf_k = w_pos (11 w_pos at k = N - 1, 0 without a goal).
`p` is any parameter block with the fields of dart_se3mpc_params (oracle.Params or _cabi.Params);
arrays are batch-first: p0, v0, goal (B, 3); T (B, 3N) thrust rows 3k+c; r, u (B, 3N)."""
from __future__ import annotations

import numpy as np


class Problems:
    """B problems of one parameter block; spheres (S, 4) [cx cy cz r], weight = obstacle_weight."""

    def __init__(self, p, p0, v0, goal=None, r=None, u=None, has_goal=None, spheres=None, weight=0.0, margin=0.0):
        self.p, self.N = p, int(p.horizon)
        N = self.N
        self.p0 = np.asarray(p0, np.float64).reshape(-1, 3)
        B = self.B = len(self.p0)
        self.v0 = np.asarray(v0, np.float64).reshape(B, 3)
        self.track = r is not None
        if self.track:
            self.r = np.asarray(r, np.float64).reshape(B, 3 * N)
            self.u = np.zeros((B, 3 * N)) if u is None else np.asarray(u, np.float64).reshape(B, 3 * N)
        else:
            self.goal = np.asarray(goal, np.float64).reshape(B, 3)
            self.r = np.tile(self.goal, (1, N))
            self.u = np.zeros((B, 3 * N))
        self.hg = np.ones(B) if has_goal is None else (np.asarray(has_goal).reshape(B) != 0).astype(np.float64)
        self.spheres = np.zeros((0, 4)) if spheres is None else np.asarray(spheres, np.float64).reshape(-1, 4)
        self.weight, self.margin = float(weight), float(margin)
        dt, m = p.dt, p.mass
        k = np.arange(N)
        D = (k[:, None] - k[None, :]).astype(np.float64)
        I3 = np.eye(3)
        # P_k = p0 + k dt v0 + sum_{j<k} dt^2 (k - j - 1/2) a_j,  V_k = v0 + sum_{j<k} dt a_j,  a = T/m - g e3
        self.Lp = np.kron(np.where(D > 0, dt * dt * (D - 0.5), 0.0), I3)
        self.Lv = np.kron(np.where(D > 0, dt, 0.0), I3)
        self.Sp = np.tile(I3, (N, 1))                       # dP/dp0 = dV/dv0
        self.Spv = np.kron((k * dt)[:, None], I3)           # dP/dv0
        last = np.zeros(N)
        last[-1] = 10.0
        self.wfac = self.hg[:, None] * np.repeat(1.0 + last, 3)[None, :]   # wpf / w_pos per entry (B, 3N)
        self.ge3 = np.tile([0.0, 0.0, p.gravity], N)
        self.hover = np.tile([0.0, 0.0, p.mass * p.gravity], N)

    # ---- the objective at thrusts T (B, 3N) ----
    def states(self, T):
        a = T / self.p.mass - self.ge3
        P = self.p0 @ self.Sp.T + self.v0 @ self.Spv.T + a @ self.Lp.T
        V = self.v0 @ self.Sp.T + a @ self.Lv.T
        return P, V, a

    def _spheres(self, P):
        """penalty (B,), gradient (B, 3N) and Hessian blocks (B, N, 3, 3) on the positions"""
        B, N = self.B, self.N
        Pk = P.reshape(B, N, 1, 3)
        c, R = self.spheres[None, None, :, :3], self.spheres[None, None, :, 3] + self.margin
        e = Pk - c
        h = R * R - (e * e).sum(-1)
        on = h > 0
        w = self.weight
        f = (w * np.where(on, h * h, 0.0)).sum((1, 2))
        g = (np.where(on, -4 * w * h, 0.0)[..., None] * e).sum(2).reshape(B, 3 * N)
        Hs = (np.where(on, 8 * w, 0.0)[..., None, None] * e[..., :, None] * e[..., None, :]
              - np.where(on, 4 * w * h, 0.0)[..., None, None] * np.eye(3)).sum(2)
        return f, g, Hs

    def fg(self, T):
        p = self.p
        P, V, a = self.states(T)
        e, ev, dev = P - self.r, V - self.u, T - self.hover
        fs, gs, _ = self._spheres(P)
        f = (p.w_pos * self.wfac * e * e).sum(1) + p.w_vel * (ev * ev).sum(1) + p.w_acc * (a * a).sum(1) \
            + p.w_thrust * (dev * dev).sum(1) + fs
        gP = 2 * p.w_pos * self.wfac * e + gs
        gV = 2 * p.w_vel * ev
        g = gP @ self.Lp / p.mass + gV @ self.Lv / p.mass + 2 * p.w_acc * a / p.mass + 2 * p.w_thrust * dev
        return f, g

    def hessian(self, T):
        p = self.p
        P, _, _ = self.states(T)
        _, _, Hs = self._spheres(P)
        B, N = self.B, self.N
        Hst = np.zeros((B, 3 * N, 3 * N))
        for k in range(N):
            Hst[:, 3 * k:3 * k + 3, 3 * k:3 * k + 3] = Hs[:, k]
        Hst += np.einsum("bi,ij->bij", 2 * p.w_pos * self.wfac, np.eye(3 * N))
        Mp, Mv = self.Lp / p.mass, self.Lv / p.mass
        H = np.einsum("ki,bkl,lj->bij", Mp, Hst, Mp) + 2 * p.w_vel * (Mv.T @ Mv)[None] \
            + (2 * p.w_acc / p.mass ** 2 + 2 * p.w_thrust) * np.eye(3 * N)[None]
        return H, Hst

    def active(self, T):
        p, N = self.p, self.N
        lo = np.tile([-p.tilt_thrust, -p.tilt_thrust, p.min_thrust], N)
        hi = np.tile([p.tilt_thrust, p.tilt_thrust, p.max_thrust], N)
        return (T == lo) | (T == hi)

    # ---- the VJP ----
    def theta_size(self):
        return 6 + (6 * self.N if self.track else 3) + 4

    def jacobians(self, T):
        """dg/dtheta (B, 3N, K), df/dtheta (B, K), direct dx/dtheta (9N, K) with theta = [p0 v0 (goal | r u) w]."""
        p, N, B = self.p, self.N, self.B
        P, V, a = self.states(T)
        e, ev, dev = P - self.r, V - self.u, T - self.hover
        _, gs, _ = self._spheres(P)
        _, Hst = self.hessian(T)
        Mp, Mv = self.Lp / p.mass, self.Lv / p.mass
        Wp = 2 * p.w_pos * self.wfac
        gP, gV = Wp * e + gs, 2 * p.w_vel * ev
        cols, fcols = [], []
        MpH = np.einsum("ki,bkl->bil", Mp, Hst)
        cols.append(MpH @ self.Sp)
        fcols.append(gP @ self.Sp)
        cols.append(MpH @ self.Spv + 2 * p.w_vel * (Mv.T @ self.Sp)[None])
        fcols.append(gP @ self.Spv + gV @ self.Sp)
        if self.track:
            cols.append(-Mp.T[None] * Wp[:, None, :])
            fcols.append(-Wp * e)
            cols.append(np.broadcast_to(-2 * p.w_vel * Mv.T, (B, 3 * N, 3 * N)))
            fcols.append(-2 * p.w_vel * ev)
        else:
            cols.append(-(Mp.T[None] * Wp[:, None, :]) @ self.Sp)
            fcols.append((-Wp * e) @ self.Sp)
        cols.append(np.stack([(2 * self.wfac * e) @ Mp, (2 * ev) @ Mv, 2 * a / p.mass, 2 * dev], axis=2))
        fcols.append(np.stack([(self.wfac * e * e).sum(1), (ev * ev).sum(1), (a * a).sum(1), (dev * dev).sum(1)], 1))
        G = np.concatenate(cols, axis=2)
        df = np.concatenate(fcols, axis=1)
        K = G.shape[2]
        Dx = np.zeros((9 * N, K))
        Dx[:3 * N, 0:3] = self.Sp
        Dx[:3 * N, 3:6] = self.Spv
        Dx[3 * N:6 * N, 3:6] = self.Sp
        return G, df, Dx

    def rollout_matrix(self):
        """d[P | V | T]/dT (9N, 3N)"""
        N, m = self.N, self.p.mass
        return np.concatenate([self.Lp / m, self.Lv / m, np.eye(3 * N)])

    def plan_jacobian(self, T):
        """(dx/dtheta (B, 9N, K), dcost/dtheta (B, K), status (B,)): the active set held, H_FF solved densely;
        status 1 where H_FF is not positive definite."""
        N = self.N
        H, _ = self.hessian(T)
        _, g = self.fg(T)
        G, df, Dx = self.jacobians(T)
        F = (~self.active(T)).astype(np.float64)
        Hm = F[:, :, None] * H * F[:, None, :] + np.einsum("bi,ij->bij", 1.0 - F, np.eye(3 * N))
        status = np.where(np.linalg.eigvalsh(Hm).min(1) > 0, 0, 1).astype(np.int32)
        Hm[status != 0] = np.eye(3 * N)
        dT = np.linalg.solve(Hm, -F[:, :, None] * G)
        dx = np.einsum("ij,bjk->bik", self.rollout_matrix(), dT) + Dx[None]
        dc = np.einsum("bi,bik->bk", g, dT) + df
        return dx, dc, status

    def vjp(self, T, gx=None, gcost=None):
        """dict(gp0, gv0, ggoal | gref, gw, status) in the layout of dart_se3mpc_solve_vjp_batch (batch-first;
        gref (B, 6N) rows 3k+c then 3N+3k+c).  Status 1 is a property of the system the entry solves,
        H_FF lam_F = tbar_F: where tbar_F is exactly zero, lam = 0 solves it whatever H_FF is (the entry runs no
        conjugate-gradient step), and the status is 0."""
        N, B = self.N, self.B
        dx, dc, status = self.plan_jacobian(T)
        gx = np.zeros((B, 9 * N)) if gx is None else np.asarray(gx, np.float64).reshape(B, 9 * N)
        gcost = np.zeros(B) if gcost is None else np.asarray(gcost, np.float64).reshape(B)
        tbar = gx @ self.rollout_matrix() + gcost[:, None] * self.fg(T)[1]
        status = np.where((tbar * ~self.active(T) == 0).all(1), 0, status).astype(np.int32)
        # where tbar_F = 0, tbar . dT/dtheta = 0 for any dT that is 0 on A: th is exact even if H_FF is singular
        th = np.einsum("bi,bik->bk", gx, dx) + gcost[:, None] * dc
        th[status != 0] = np.nan
        out = dict(gp0=th[:, 0:3], gv0=th[:, 3:6], gw=th[:, -4:], status=status)
        if self.track:
            out["gref"] = th[:, 6:6 + 6 * N]
        else:
            out["ggoal"] = th[:, 6:9]
        return out
