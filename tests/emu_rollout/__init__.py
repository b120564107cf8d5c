"""Host emulation of the kernel core in the dynamics-consistent modes (tests only; see
emu_rollout.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libemu_rollout.so")
_SRCS = [os.path.join(_HERE, "emu_rollout.cpp"),
         os.path.join(_HERE, "..", "..", "dart_planner_b200", "csrc", "se3mpc_core.cuh"),
         os.path.join(_HERE, "..", "..", "include", "dart_se3mpc.h")]
_lib = None


def build(force=False):
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in _SRCS):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", _LIB, _SRCS[0]],
                       check=True)
    return _LIB


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB)
    return _lib


def set_policy(policy):
    """"latency" (register-rich build), "throughput" (register-capped build) or "two-phase" (the
    throughput build's context switch after the first iteration)."""
    lib().emr_set_ls_shared(1 if policy in ("throughput", "two-phase") else 0)
    lib().emr_set_two_phase(1 if policy == "two-phase" else 0)


class Result:
    pass


def solve_batch(params, p0, v0, goal, has_goal=None, x_warm=None, grid=None):
    """params: dart_planner_b200._cabi.Params with gradient_mode 3 or 4 (4 needs grid: _cabi.Grid)."""
    p0 = np.ascontiguousarray(p0, np.float64).reshape(-1, 3)
    B = len(p0)
    v0 = np.ascontiguousarray(v0, np.float64).reshape(B, 3)
    goal = np.ascontiguousarray(goal, np.float64).reshape(B, 3)
    N = params.horizon
    r = Result()
    r.x = np.zeros((B, 9 * N)); r.cost = np.zeros(B)
    r.nit = np.zeros(B, np.int32); r.nfev = np.zeros(B, np.int32)
    r.status = np.zeros(B, np.int32); r.task = np.zeros(B, np.int32)
    r.accelerations = np.zeros((B, N, 3)); r.attitudes = np.zeros((B, N, 3))
    r.body_rates = np.zeros((B, N, 3)); r.thrusts = np.zeros((B, N))
    hg = None if has_goal is None else np.ascontiguousarray(has_goal, np.uint8)
    xw = None if x_warm is None else np.ascontiguousarray(x_warm, np.float64).reshape(B, 9 * N)
    vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    rc = lib().emr_solve_batch(C.byref(params), C.c_long(B), vp(p0), vp(v0), vp(goal), vp(hg), vp(xw), vp(r.x),
                               vp(r.cost), vp(r.nit), vp(r.nfev), vp(r.status), vp(r.task), vp(r.accelerations),
                               vp(r.attitudes), vp(r.body_rates), vp(r.thrusts), None if grid is None else C.byref(grid))
    if rc != 0:
        raise RuntimeError(f"emr_solve_batch: {rc}")
    return r
