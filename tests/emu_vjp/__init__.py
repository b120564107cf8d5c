"""Host emulation of the differentiable solve's device routine (tests only; see emu_vjp.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libemu_vjp.so")
_SRCS = [os.path.join(_HERE, "emu_vjp.cpp"),
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


def vjp_batch(params, p0, v0, goal, x, gx=None, gcost=None, ref=None, spheres=None, margin=0.0, has_goal=None):
    """The arguments of dart_se3mpc_solve_vjp_batch in batch-first host arrays: p0, v0, goal (B, 3);
    x, gx (B, 9N); gcost (B,); ref (B, 6N) (each problem's column of the reference block) or None;
    spheres (S, 4).  Returns dict(gp0, gv0, ggoal (B, 3), gref (B, 6N), gw (B, 4), status (B,))."""
    N = params.horizon
    p0 = np.asarray(p0, np.float64).reshape(-1, 3)
    B = len(p0)
    soa = lambda a, rows: None if a is None else np.ascontiguousarray(np.asarray(a, np.float64).reshape(B, rows).T)  # noqa: E731
    ins = dict(p0=soa(p0, 3), v0=soa(v0, 3), goal=soa(goal if goal is not None else np.zeros((B, 3)), 3),
               x=soa(x, 9 * N), gx=soa(gx, 9 * N), gcost=None if gcost is None else np.ascontiguousarray(gcost, np.float64),
               ref=soa(ref, 6 * N))
    s = None if spheres is None else np.ascontiguousarray(spheres, np.float64).reshape(-1, 4)
    hg = None if has_goal is None else np.ascontiguousarray(has_goal, np.uint8)
    out = dict(gp0=np.zeros((3, B)), gv0=np.zeros((3, B)), ggoal=np.zeros((3, B)), gref=np.zeros((6 * N, B)),
               gw=np.zeros((4, B)), status=np.zeros(B, np.int32))
    vp = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    rc = lib().emv_vjp_batch(C.byref(params), C.c_long(B), C.c_long(B), vp(ins["p0"]), vp(ins["v0"]), vp(ins["goal"]),
                             vp(hg), vp(ins["x"]), vp(ins["ref"]), vp(s) if s is not None and len(s) else None,
                             C.c_int(0 if s is None else len(s)), C.c_double(margin), vp(ins["gx"]), vp(ins["gcost"]),
                             vp(out["gp0"]), vp(out["gv0"]), vp(out["ggoal"]), vp(out["gref"]), vp(out["gw"]),
                             vp(out["status"]))
    if rc != 0:
        raise RuntimeError(f"emv_vjp_batch: {rc}")
    return {k: (v if k == "status" else v.T.copy()) for k, v in out.items()}
