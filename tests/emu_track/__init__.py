"""Host emulation of the kernel core in the tracking modes 7 and 8 (tests only; see emu_track.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libemu_track.so")
_SRCS = [os.path.join(_HERE, "emu_track.cpp"),
         os.path.join(_HERE, "..", "..", "dart_planner_b200", "csrc", "se3mpc_core.cuh"),
         os.path.join(_HERE, "..", "..", "include", "dart_se3mpc.h")]
_lib = None

POLICIES = ("latency", "throughput", "two-phase")


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
    assert policy in POLICIES, policy
    lib().emt_set_policy(1 if policy in ("throughput", "two-phase") else 0, 1 if policy == "two-phase" else 0)


class Result:
    pass


def ref_columns(P, V, B):
    """(P (B, T, 3), V (B, T, 3) or None) -> (B, 6T): each problem's column of the dart_track_ref block."""
    P = np.ascontiguousarray(P, np.float64).reshape(B, -1, 3)
    V = np.zeros_like(P) if V is None else np.ascontiguousarray(V, np.float64).reshape(P.shape)
    return np.ascontiguousarray(np.concatenate([P.reshape(B, -1), V.reshape(B, -1)], axis=1)), P.shape[1]


def solve_batch(params, p0, v0, ref, start=0, spheres=None, margin=0.0, has_goal=None, x_warm=None):
    """params: dart_planner_b200._cabi.Params with gradient_mode 7 or 8; ref = (P, V or None)."""
    p0 = np.ascontiguousarray(p0, np.float64).reshape(-1, 3)
    B = len(p0)
    v0 = np.ascontiguousarray(v0, np.float64).reshape(B, 3)
    cols, T = ref_columns(ref[0], ref[1], B)
    s = np.zeros((0, 4)) if spheres is None else np.ascontiguousarray(spheres, np.float64).reshape(-1, 4)
    N = params.horizon
    r = Result()
    r.x = np.zeros((B, 9 * N)); r.cost = np.zeros(B)
    r.nit = np.zeros(B, np.int32); r.nfev = np.zeros(B, np.int32)
    r.status = np.zeros(B, np.int32); r.task = np.zeros(B, np.int32)
    r.accelerations = np.zeros((B, N, 3)); r.attitudes = np.zeros((B, N, 3))
    r.body_rates = np.zeros((B, N, 3)); r.thrusts = np.zeros((B, N))
    hg = None if has_goal is None else np.ascontiguousarray(has_goal, np.uint8)
    xw = None if x_warm is None else np.ascontiguousarray(x_warm, np.float64).reshape(B, 9 * N)
    vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = lib().emt_solve_batch(C.byref(params), C.c_long(B), vp(p0), vp(v0), vp(hg), vp(xw), vp(cols), C.c_int(T),
                               C.c_int(start), vp(s) if len(s) else None, C.c_int(len(s)), C.c_double(margin),
                               vp(r.x), vp(r.cost), vp(r.nit), vp(r.nfev), vp(r.status), vp(r.task),
                               vp(r.accelerations), vp(r.attitudes), vp(r.body_rates), vp(r.thrusts))
    if rc != 0:
        raise RuntimeError(f"emt_solve_batch: {rc}")
    return r
