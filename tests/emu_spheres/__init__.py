"""Host emulation of the kernel core in the sphere-penalty modes 5 and 6 (tests only; see
emu_spheres.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libemu_spheres.so")
_SRCS = [os.path.join(_HERE, "emu_spheres.cpp"),
         os.path.join(_HERE, "..", "..", "dart_planner_b200", "csrc", "se3mpc_core.cuh"),
         os.path.join(_HERE, "..", "..", "include", "dart_se3mpc.h")]
_lib = None

POLICIES = {5: ("latency", "throughput", "seven-slot", "two-phase"), 6: ("latency", "throughput", "two-phase")}


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
    """"latency" (register-rich build), "throughput" (register-capped build), "seven-slot" (mode 5:
    the TILT=false instantiation, latency build) or "two-phase" (the throughput build's context
    switch after the first iteration)."""
    assert policy in ("latency", "throughput", "seven-slot", "two-phase"), policy
    lib().ems_set_policy(1 if policy in ("throughput", "two-phase") else 0, 1 if policy == "two-phase" else 0,
                         1 if policy == "seven-slot" else 0)


class Result:
    pass


def penalty(spheres, P, weight, margin):
    """(f (npos,), grad (npos, 3)) of the core's SpherePenalty at positions P (npos, 3)."""
    s = np.ascontiguousarray(spheres, np.float64).reshape(-1, 4)
    P = np.ascontiguousarray(P, np.float64).reshape(-1, 3)
    f, g = np.zeros(len(P)), np.zeros((len(P), 3))
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    lib().ems_penalty(vp(s), C.c_int(len(s)), C.c_double(weight), C.c_double(margin), C.c_long(len(P)), vp(P),
                      vp(f), vp(g))
    return f, g


def solve_batch(params, p0, v0, goal, spheres, margin, has_goal=None, x_warm=None):
    """params: dart_planner_b200._cabi.Params with gradient_mode 5 or 6; spheres (S, 4)."""
    p0 = np.ascontiguousarray(p0, np.float64).reshape(-1, 3)
    B = len(p0)
    v0 = np.ascontiguousarray(v0, np.float64).reshape(B, 3)
    goal = np.ascontiguousarray(goal, np.float64).reshape(B, 3)
    s = np.ascontiguousarray(spheres, np.float64).reshape(-1, 4)
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
    rc = lib().ems_solve_batch(C.byref(params), C.c_long(B), vp(p0), vp(v0), vp(goal), vp(hg), vp(xw),
                               vp(s) if len(s) else None, C.c_int(len(s)), C.c_double(margin), vp(r.x), vp(r.cost),
                               vp(r.nit), vp(r.nfev), vp(r.status), vp(r.task), vp(r.accelerations),
                               vp(r.attitudes), vp(r.body_rates), vp(r.thrusts))
    if rc != 0:
        raise RuntimeError(f"ems_solve_batch: {rc}")
    return r
