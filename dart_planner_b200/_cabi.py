"""ctypes binding of the C-ABI shared library (include/dart_se3mpc.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``dart_planner_b200.build``.
There is no CPU fallback: if the library is missing or no CUDA device is present the calls
raise.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DART_SE3MPC_LIB") or os.path.join(_HERE, "lib", "libdart_se3mpc.so")  # env: A/B builds

DART_OK, DART_E_BADARG, DART_E_UNSUPPORTED, DART_E_CUDA, DART_E_NODEVICE = 0, -1, -2, -3, -4
TASK_NAMES = {
    0: "START",
    1: "CONVERGENCE: NORM OF PROJECTED GRADIENT <= PGTOL",
    2: "CONVERGENCE: RELATIVE REDUCTION OF F <= FACTR*EPSMCH",
    3: "STOP: TOTAL NO. OF ITERATIONS REACHED LIMIT",
    4: "STOP: TOTAL NO. OF F,G EVALUATIONS EXCEEDS LIMIT",
    5: "ABNORMAL: ",
}


class Params(C.Structure):
    """Mirror of ``dart_se3mpc_params`` (include/dart_se3mpc.h)."""

    _fields_ = [
        ("struct_size", C.c_int32), ("horizon", C.c_int32), ("max_iterations", C.c_int32),
        ("max_corrections", C.c_int32), ("max_linesearch", C.c_int32), ("max_fun", C.c_int32),
        ("gradient_mode", C.c_int32), ("reserved0", C.c_int32),
        ("dt", C.c_double), ("mass", C.c_double), ("gravity", C.c_double),
        ("pos_bound", C.c_double), ("max_velocity", C.c_double), ("tilt_thrust", C.c_double),
        ("min_thrust", C.c_double), ("max_thrust", C.c_double),
        ("w_pos", C.c_double), ("w_vel", C.c_double), ("w_acc", C.c_double),
        ("w_thrust", C.c_double), ("gtol", C.c_double), ("ftol", C.c_double),
        ("w_obstacle", C.c_double), ("obstacle_free_level", C.c_double),
    ]


class Grid(C.Structure):
    """Mirror of ``dart_grid``."""

    _fields_ = [
        ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32),
        ("ox", C.c_int32), ("oy", C.c_int32), ("oz", C.c_int32),
        ("resolution", C.c_double), ("prior", C.c_double), ("occ", C.c_void_p),
        ("cell_bytes", C.c_int32), ("reserved", C.c_int32),
    ]


class Spheres(C.Structure):
    """Mirror of ``dart_spheres``: the sphere list of gradient_mode 5 / 6."""

    _fields_ = [
        ("n", C.c_int32), ("reserved", C.c_int32), ("cxyzr", C.c_void_p), ("margin", C.c_double),
    ]


class TrackRef(C.Structure):
    """Mirror of ``dart_track_ref``: the per-timestep reference of gradient_mode 7 / 8."""

    _fields_ = [("len", C.c_int32), ("start", C.c_int32), ("rows", C.c_void_p)]


EXPORTS = [
    "dart_abi_version", "dart_last_cuda_error", "dart_se3mpc_default_params",
    "dart_se3mpc_solve_batch", "dart_se3mpc_solve_batch_map", "dart_se3mpc_closed_loop_step",
    "dart_se3mpc_solve_batch_host", "dart_se3mpc_release_thread_workspace", "dart_se3mpc_row_stride", "dart_se3mpc_solve_batch_rows", "dart_se3mpc_extract_batch",
    "dart_launch_count", "dart_se3mpc_set_inflight_hint",
    "dart_se3mpc_kernel_info", "dart_map_query_batch", "dart_map_traj_safe_batch",
    "dart_map_trace_ray_batch", "dart_map_update_batch", "dart_map_add_spheres", "dart_fp64_probe", "dart_ddiv_selftest",
    "dart_map_signed_distance", "dart_map_clearance_field", "dart_se3mpc_closed_loop_step_map",
    "dart_se3mpc_solve_batch_spheres", "dart_se3mpc_solve_batch_host_spheres", "dart_se3mpc_closed_loop_step_spheres",
    "dart_se3mpc_solve_batch_track", "dart_se3mpc_closed_loop_step_track", "dart_se3mpc_solve_vjp_batch",
]

_lib = None


class LibraryMissing(RuntimeError):
    pass


def lib():
    """Load the CUDA library; fail loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). dart_planner_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    L.dart_abi_version.restype = C.c_int
    L.dart_last_cuda_error.restype = C.c_char_p
    L.dart_se3mpc_default_params.argtypes = [C.POINTER(Params)]
    L.dart_se3mpc_default_params.restype = None
    L.dart_se3mpc_solve_batch.argtypes = [C.POINTER(Params), i64, i64] + [vp] * 16 + [vp]
    L.dart_se3mpc_solve_batch.restype = C.c_int
    L.dart_se3mpc_solve_batch_map.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 16 +
                                              [C.POINTER(Grid), C.c_double, C.c_double, vp, vp])
    L.dart_se3mpc_solve_batch_map.restype = C.c_int
    L.dart_se3mpc_closed_loop_step.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 5 + [i32] +
                                               [vp] * 4 + [C.c_double, vp])
    L.dart_se3mpc_closed_loop_step.restype = C.c_int
    L.dart_se3mpc_closed_loop_step_map.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 5 + [i32] +
                                                   [vp] * 4 + [C.c_double, C.POINTER(Grid), C.POINTER(Grid),
                                                                C.c_double, C.c_double, i32, vp, vp])
    L.dart_se3mpc_closed_loop_step_map.restype = C.c_int
    L.dart_se3mpc_solve_batch_host.argtypes = [C.POINTER(Params), i64] + [vp] * 14
    L.dart_se3mpc_solve_batch_host.restype = C.c_int
    L.dart_se3mpc_solve_batch_spheres.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 16 +
                                                  [C.POINTER(Spheres), C.POINTER(Grid), C.c_double, C.c_double,
                                                   vp, vp])
    L.dart_se3mpc_solve_batch_spheres.restype = C.c_int
    L.dart_se3mpc_solve_batch_host_spheres.argtypes = [C.POINTER(Params), i64] + [vp] * 14 + [C.POINTER(Spheres)]
    L.dart_se3mpc_solve_batch_host_spheres.restype = C.c_int
    L.dart_se3mpc_closed_loop_step_spheres.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 5 + [i32] +
                                                       [vp] * 4 + [C.c_double, C.POINTER(Spheres), C.POINTER(Grid),
                                                                    C.c_double, C.c_double, i32, vp, vp])
    L.dart_se3mpc_closed_loop_step_spheres.restype = C.c_int
    L.dart_se3mpc_solve_batch_track.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 15 +
                                                 [C.POINTER(TrackRef), C.POINTER(Spheres), C.POINTER(Grid),
                                                  C.c_double, C.c_double, vp, vp])
    L.dart_se3mpc_solve_batch_track.restype = C.c_int
    L.dart_se3mpc_closed_loop_step_track.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 4 + [i32] +
                                                     [vp] * 4 + [C.c_double, C.POINTER(TrackRef), C.POINTER(Spheres),
                                                                  C.POINTER(Grid), C.c_double, C.c_double, i32, vp, vp])
    L.dart_se3mpc_closed_loop_step_track.restype = C.c_int
    L.dart_se3mpc_solve_vjp_batch.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 5 + [C.POINTER(TrackRef),
                                              C.POINTER(Spheres)] + [vp] * 9)
    L.dart_se3mpc_solve_vjp_batch.restype = C.c_int
    L.dart_se3mpc_extract_batch.argtypes = [C.POINTER(Params), i64, i64] + [vp] * 5 + [i32, vp]
    L.dart_se3mpc_extract_batch.restype = C.c_int
    L.dart_se3mpc_release_thread_workspace.argtypes = []
    L.dart_se3mpc_release_thread_workspace.restype = None
    L.dart_se3mpc_row_stride.argtypes = [C.POINTER(Params), i32]
    L.dart_se3mpc_row_stride.restype = C.c_int64
    L.dart_se3mpc_solve_batch_rows.argtypes = ([C.POINTER(Params), i64, i64] + [vp] * 7 + [i64, i32] +
                                               [C.POINTER(Grid), C.c_double, C.c_double, i32, vp])
    L.dart_se3mpc_solve_batch_rows.restype = C.c_int
    L.dart_launch_count.restype = C.c_int64
    L.dart_se3mpc_set_inflight_hint.argtypes = [i64]
    L.dart_se3mpc_set_inflight_hint.restype = C.c_int
    L.dart_se3mpc_kernel_info.argtypes = [C.POINTER(Params), i64] + [C.POINTER(i32)] * 5
    L.dart_se3mpc_kernel_info.restype = C.c_int
    L.dart_map_query_batch.argtypes = [C.POINTER(Grid), i64, i64, vp, vp, vp]
    L.dart_map_query_batch.restype = C.c_int
    L.dart_map_traj_safe_batch.argtypes = [C.POINTER(Grid), i64, i64, i32, vp, C.c_double,
                                           C.c_double, vp, vp]
    L.dart_map_traj_safe_batch.restype = C.c_int
    L.dart_map_trace_ray_batch.argtypes = [C.c_double, i64, i64, vp, vp, vp, i32, vp, vp, vp]
    L.dart_map_trace_ray_batch.restype = C.c_int
    L.dart_map_update_batch.argtypes = [C.POINTER(Grid), vp, vp, i64, i64, vp, vp, vp, vp, C.c_double,
                                        C.c_double, C.c_double, vp, vp]
    L.dart_map_update_batch.restype = C.c_int
    L.dart_map_add_spheres.argtypes = [C.POINTER(Grid), vp, i32, vp, vp, C.c_double, vp]
    L.dart_map_add_spheres.restype = C.c_int
    L.dart_map_signed_distance.argtypes = [C.POINTER(Grid), C.c_double, vp, vp, vp]
    L.dart_map_signed_distance.restype = C.c_int
    L.dart_map_clearance_field.argtypes = [C.POINTER(Grid), C.c_double, C.c_double, C.c_double, vp, vp, vp]
    L.dart_map_clearance_field.restype = C.c_int
    L.dart_fp64_probe.argtypes = [i32, C.POINTER(i32), vp, vp]
    L.dart_fp64_probe.restype = C.c_int
    L.dart_ddiv_selftest.argtypes = [i64, C.c_uint64, i32, vp, vp]
    L.dart_ddiv_selftest.restype = C.c_int
    if L.dart_abi_version() != 1:
        raise RuntimeError("libdart_se3mpc.so ABI version mismatch")
    _lib = L
    return _lib


def check(rc: int, what: str):
    if rc == DART_OK:
        return
    L = lib()
    detail = L.dart_last_cuda_error().decode() if rc == DART_E_CUDA else ""
    names = {-1: "bad argument", -2: "unsupported configuration", -3: "CUDA error",
             -4: "no CUDA device"}
    raise RuntimeError(f"{what} failed: {names.get(rc, rc)} {detail}".strip())
