"""ctypes binding of the CPU oracle of the sphere obstacle penalty (sphere_oracle.c) -- TEST
INFRASTRUCTURE, NOT PRODUCT CODE.  gradient_mode 5 (mode 0 + spheres) on the reference oracle's
driver, gradient_mode 6 (mode 3 + spheres) on the dynamics-consistent oracle's rollout and adjoint.
Parameters and the result type are the reference oracle's (``oracle``)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(_HERE, "..", "..", "oracle")
_LIB_PATH = os.path.join(_HERE, "libsphere_oracle.so")
_SRCS = [os.path.join(_HERE, "sphere_oracle.c"), os.path.join(_HERE, "..", "rollout_oracle", "rollout_oracle.c"),
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
        L.sph_solve_batch.argtypes = [PP, C.c_int, C.c_int64, dp, dp, dp, u8p, dp, dp, C.c_int32, C.c_double,
                                      C.c_double, dp, dp, ip, ip, ip, ip, dp, dp, dp, dp, C.c_int]
        L.sph_solve_batch.restype = C.c_int
        L.sph_penalty_batch.argtypes = [dp, C.c_int32, C.c_double, C.c_double, C.c_int64, dp, dp, dp]
        L.sph_penalty_batch.restype = C.c_double
        L.sph_fg.argtypes = [PP, C.c_int, dp, dp, dp, dp, C.c_int32, C.c_double, C.c_double, dp, dp, dp]
        L.sph_fg.restype = C.c_double
        _lib = L
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _c(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


def sphere_list(centers, radii):
    """(S, 4) [cx cy cz r], the layout of dart_spheres."""
    c = _c(centers).reshape(-1, 3)
    return np.ascontiguousarray(np.concatenate([c, _c(radii).reshape(-1, 1)], axis=1))


def penalty(spheres, P, weight, margin):
    """(f (npos,), grad (npos, 3)) of the sphere penalty at positions P (npos, 3)."""
    s = _c(spheres).reshape(-1, 4)
    P = _c(P).reshape(-1, 3)
    f, g = np.zeros(len(P)), np.zeros((len(P), 3))
    lib().sph_penalty_batch(_dp(s), len(s), float(weight), float(margin), len(P), _dp(P), _dp(f), _dp(g))
    return f, g


def fg(p: oracle.Params, mode, p0, v0, goal, v, spheres, weight, margin):
    """Mode 5: (f, g) at the packed x (9N).  Mode 6: (f, df/dT) at the thrusts T (3N)."""
    N = p.horizon
    s = _c(spheres).reshape(-1, 4)
    v = _c(v).ravel()
    g, xs = np.zeros_like(v), np.zeros(9 * N)
    f = lib().sph_fg(C.byref(p), int(mode), _dp(_c(p0)), _dp(_c(v0)), _dp(None if goal is None else _c(goal)),
                     _dp(s), len(s), float(weight), float(margin), _dp(v), _dp(xs), _dp(g))
    return f, g


def solve_batch(p: oracle.Params, mode, p0, v0, goal, spheres, weight, margin, has_goal=None, x_warm=None,
                nthreads=1) -> oracle.BatchResult:
    """gradient_mode 5 or 6 for B problems with one shared (S, 4) sphere list."""
    p0 = _c(p0).reshape(-1, 3)
    B = p0.shape[0]
    v0, goal = _c(v0, (B, 3)), _c(goal, (B, 3))
    N = p.horizon
    s = _c(spheres).reshape(-1, 4)
    hg = None if has_goal is None else np.ascontiguousarray(has_goal, np.uint8).reshape(B)
    xw = None if x_warm is None else _c(x_warm, (B, 9 * N))
    x, cost = np.zeros((B, 9 * N)), np.zeros(B)
    nit, nfev, status, task = (np.zeros(B, np.int32) for _ in range(4))
    acc, att, rates, thrust = np.zeros((B, N, 3)), np.zeros((B, N, 3)), np.zeros((B, N, 3)), np.zeros((B, N))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))  # noqa: E731
    rc = lib().sph_solve_batch(C.byref(p), int(mode), B, _dp(p0), _dp(v0), _dp(goal),
                               None if hg is None else hg.ctypes.data_as(C.POINTER(C.c_uint8)), _dp(xw), _dp(s),
                               len(s), float(weight), float(margin), _dp(x), _dp(cost), ip(nit), ip(nfev),
                               ip(status), ip(task), _dp(acc), _dp(att), _dp(rates), _dp(thrust), int(nthreads))
    if rc != 0:
        raise RuntimeError(f"sph_solve_batch failed: {rc}")
    return oracle.BatchResult(x, cost, nit, nfev, status, task, acc, att, rates, thrust, 0.0)
