"""ctypes binding of the CPU oracle of reference tracking (track_oracle.c) -- TEST INFRASTRUCTURE,
NOT PRODUCT CODE.  gradient_mode 7 (mode 3 tracking a per-timestep reference) and 8 (mode 6 tracking
it) on the reference oracle's driver over the 3N thrusts.  Parameters and the result type are the
reference oracle's (``oracle``).  A reference is (P (B, T, 3), V (B, T, 3)); timestep k of a solve
tracks sample min(start + k, T - 1)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(_HERE, "..", "..", "oracle")
_LIB_PATH = os.path.join(_HERE, "libtrack_oracle.so")
_SRCS = [os.path.join(_HERE, "track_oracle.c"), os.path.join(_HERE, "..", "sphere_oracle", "sphere_oracle.c"),
         os.path.join(_HERE, "..", "rollout_oracle", "rollout_oracle.c"),
         os.path.join(_ORACLE, "se3mpc_oracle.c"), os.path.join(_ORACLE, "lbfgsb_oracle.c")]
_lib = None


def build(force: bool = False) -> str:
    deps = _SRCS + [os.path.join(_ORACLE, "se3mpc_oracle.h")]
    if force or not os.path.exists(_LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in deps):
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=c11", "-Wall", "-Wextra", "-ffp-contract=off", "-fno-fast-math",
                        "-shared", "-o", _LIB_PATH] + _SRCS + ["-lm", "-lpthread"], check=True)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        dp, ip, u8p, PP = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.POINTER(oracle.Params)
        i32, f8 = C.c_int32, C.c_double
        L.trk_solve_batch.argtypes = [PP, C.c_int, C.c_int64, dp, dp, u8p, dp, dp, dp, i32, i32, dp, i32, f8, f8,
                                      dp, dp, ip, ip, ip, ip, dp, dp, dp, dp, C.c_int]
        L.trk_solve_batch.restype = C.c_int
        L.trk_fg_one.argtypes = [PP, C.c_int, dp, dp, C.c_int, dp, dp, i32, i32, dp, i32, f8, f8, dp, dp, dp]
        L.trk_fg_one.restype = C.c_double
        _lib = L
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _c(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


def _ref(P, V, B):
    P = _c(P)
    P = P.reshape(B, -1, 3)
    V = np.zeros_like(P) if V is None else _c(V, P.shape)
    return P, V


def fg(p: oracle.Params, mode, p0, v0, ref, T_thrust, spheres=None, weight=0.0, margin=0.0, start=0, has_goal=True):
    """(f, df/dT) of mode 7 / 8 at the thrusts (3N) of one problem; ref = (P (T, 3), V (T, 3) or None)."""
    N = p.horizon
    P, V = _ref(ref[0], ref[1], 1)
    s = np.zeros((0, 4)) if spheres is None else _c(spheres).reshape(-1, 4)
    t = _c(T_thrust).ravel()
    g, xs = np.zeros(3 * N), np.zeros(9 * N)
    f = lib().trk_fg_one(C.byref(p), int(mode), _dp(_c(p0)), _dp(_c(v0)), 1 if has_goal else 0, _dp(P), _dp(V),
                         P.shape[1], int(start), _dp(s), len(s), float(weight), float(margin), _dp(t), _dp(xs), _dp(g))
    return f, g


def solve_batch(p: oracle.Params, mode, p0, v0, ref, start=0, spheres=None, weight=0.0, margin=0.0, has_goal=None,
                x_warm=None, nthreads=1) -> oracle.BatchResult:
    """gradient_mode 7 or 8 for B problems; ref = (P (B, T, 3), V (B, T, 3) or None); mode 8 takes
    one shared (S, 4) sphere list."""
    p0 = _c(p0).reshape(-1, 3)
    B = p0.shape[0]
    v0 = _c(v0, (B, 3))
    P, V = _ref(ref[0], ref[1], B)
    N = p.horizon
    s = np.zeros((0, 4)) if spheres is None else _c(spheres).reshape(-1, 4)
    hg = None if has_goal is None else np.ascontiguousarray(has_goal, np.uint8).reshape(B)
    xw = None if x_warm is None else _c(x_warm, (B, 9 * N))
    x, cost = np.zeros((B, 9 * N)), np.zeros(B)
    nit, nfev, status, task = (np.zeros(B, np.int32) for _ in range(4))
    acc, att, rates, thrust = np.zeros((B, N, 3)), np.zeros((B, N, 3)), np.zeros((B, N, 3)), np.zeros((B, N))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))  # noqa: E731
    rc = lib().trk_solve_batch(C.byref(p), int(mode), B, _dp(p0), _dp(v0),
                               None if hg is None else hg.ctypes.data_as(C.POINTER(C.c_uint8)), _dp(xw), _dp(P),
                               _dp(V), P.shape[1], int(start), _dp(s), len(s), float(weight), float(margin), _dp(x),
                               _dp(cost), ip(nit), ip(nfev), ip(status), ip(task), _dp(acc), _dp(att), _dp(rates),
                               _dp(thrust), int(nthreads))
    if rc != 0:
        raise RuntimeError(f"trk_solve_batch failed: {rc}")
    return oracle.BatchResult(x, cost, nit, nfev, status, task, acc, att, rates, thrust, 0.0)


def closed_loop(p: oracle.Params, mode, p0, v0, ref, steps, spheres=None, weight=0.0, margin=0.0, nthreads=16,
                record=False):
    """The closed loop of ClosedLoopSim in mode 7 / 8 with plant_dt = dt: step s solves with the
    reference window starting at sample s (warm from the previous solution after the first), and the
    state advances to the plan's P_1 / V_1 (the rollout of T_0 over one dt).  Returns (p, v, history
    (steps, B, 3) or None)."""
    N = p.horizon
    pp, vv, x = _c(p0).copy(), _c(v0).copy(), None
    hist = []
    for s in range(steps):
        x = solve_batch(p, mode, pp, vv, ref, start=s, spheres=spheres, weight=weight, margin=margin, x_warm=x,
                        nthreads=nthreads).x
        pp, vv = x[:, 3:6].copy(), x[:, 3 * N + 3:3 * N + 6].copy()
        if record:
            hist.append(pp)
    return pp, vv, (np.stack(hist) if record else None)
