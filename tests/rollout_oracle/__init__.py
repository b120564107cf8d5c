"""ctypes binding of the CPU oracle of the dynamics-consistent solve mode (rollout_oracle.c) --
TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Parameters, grids, the objective and the result type are
the reference oracle's (``oracle``); this library is built from rollout_oracle.c together with the
reference oracle's sources."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(_HERE, "..", "..", "oracle")
_LIB_PATH = os.path.join(_HERE, "librollout_oracle.so")
_SRCS = [os.path.join(_HERE, "rollout_oracle.c"), os.path.join(_ORACLE, "se3mpc_oracle.c"),
         os.path.join(_ORACLE, "lbfgsb_oracle.c")]
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
        dp, ip, u8p, PP, GP = (C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8),
                               C.POINTER(oracle.Params), C.POINTER(oracle.Grid))
        L.rol_rollout.argtypes = [PP, dp, dp, dp]
        L.rol_fg.argtypes = [PP, dp, dp, dp, GP, C.c_double, C.c_double, dp, dp, dp]
        L.rol_fg.restype = C.c_double
        L.rol_solve_batch.argtypes = [PP, C.c_int64, dp, dp, dp, u8p, dp, dp, dp, ip, ip, ip, ip, dp, dp, dp, dp,
                                      C.c_int, GP, C.c_double, C.c_double]
        L.rol_solve_batch.restype = C.c_int
        _lib = L
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _c(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if shape is None else a.reshape(shape)


def rollout(p: oracle.Params, p0, v0, T):
    """The packed x [P | V | T] whose P and V are the plant rollout of the (N, 3) thrusts T."""
    N = p.horizon
    x = np.zeros(9 * N)
    x[6 * N:] = np.asarray(T, np.float64).reshape(3 * N)
    lib().rol_rollout(C.byref(p), _dp(_c(p0)), _dp(_c(v0)), _dp(x))
    return x


def dynamics_fg(p: oracle.Params, p0, v0, goal, T, grid=None, obstacle_weight=0.0, free_level=0.5):
    """(f, df/dT) of the dynamics-consistent mode at the (N, 3) thrusts T (adjoint gradient)."""
    N = p.horizon
    x, gT = np.zeros(9 * N), np.zeros(3 * N)
    f = lib().rol_fg(C.byref(p), _dp(_c(p0)), _dp(_c(v0)), _dp(None if goal is None else _c(goal)),
                     C.byref(grid.g) if grid is not None else None, float(obstacle_weight), float(free_level),
                     _dp(_c(T, 3 * N)), _dp(x), _dp(gT))
    return f, gT


def solve_batch(p: oracle.Params, p0, v0, goal, has_goal=None, x_warm=None, nthreads=1, grid=None,
                obstacle_weight=0.0, free_level=0.5) -> oracle.BatchResult:
    """gradient_mode 3 for B problems; with grid (an ``oracle.DenseGrid``), mode 4."""
    p0 = _c(p0).reshape(-1, 3)
    B = p0.shape[0]
    v0, goal = _c(v0, (B, 3)), _c(goal, (B, 3))
    N = p.horizon
    hg = None if has_goal is None else np.ascontiguousarray(has_goal, np.uint8).reshape(B)
    xw = None if x_warm is None else _c(x_warm, (B, 9 * N))
    x, cost = np.zeros((B, 9 * N)), np.zeros(B)
    nit, nfev, status, task = (np.zeros(B, np.int32) for _ in range(4))
    acc, att, rates, thrust = np.zeros((B, N, 3)), np.zeros((B, N, 3)), np.zeros((B, N, 3)), np.zeros((B, N))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    rc = lib().rol_solve_batch(C.byref(p), B, _dp(p0), _dp(v0), _dp(goal),
                               None if hg is None else hg.ctypes.data_as(C.POINTER(C.c_uint8)), _dp(xw), _dp(x),
                               _dp(cost), ip(nit), ip(nfev), ip(status), ip(task), _dp(acc), _dp(att), _dp(rates),
                               _dp(thrust), int(nthreads), C.byref(grid.g) if grid is not None else None,
                               float(obstacle_weight), float(free_level))
    if rc != 0:
        raise RuntimeError(f"rol_solve_batch failed: {rc}")
    return oracle.BatchResult(x, cost, nit, nfev, status, task, acc, att, rates, thrust, 0.0)
