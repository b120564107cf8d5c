"""ctypes binding of the CPU oracle (oracle/*.c) -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package; ``dart_planner_b200`` never does.

Parity pinning: the oracle is checked against golden fixtures under tests/golden/ that were
produced by the UNMODIFIED reference planner (tools/gen_golden.py, SciPy 1.18.1) and, in the
build container, live against SciPy's L-BFGS-B (tests/test_oracle_vs_scipy.py).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libse3mpc_oracle.so")
_SRCS = ["se3mpc_oracle.c", "lbfgsb_oracle.c", "se3mpc_oracle.h"]


def build(force: bool = False) -> str:
    """Compile the oracle with gcc if the library is missing or stale."""
    stale = force or not os.path.exists(_LIB_PATH)
    if not stale:
        t = os.path.getmtime(_LIB_PATH)
        stale = any(os.path.getmtime(os.path.join(_HERE, s)) > t for s in _SRCS)
    if stale:
        subprocess.run(["make", "-C", _HERE, "-B", "libse3mpc_oracle.so"], check=True,
                       stdout=subprocess.DEVNULL)
    return _LIB_PATH


class Params(C.Structure):
    """Mirror of ``orc_params`` (oracle/se3mpc_oracle.h)."""

    _fields_ = [
        ("horizon", C.c_int32), ("max_iterations", C.c_int32), ("max_corrections", C.c_int32),
        ("max_linesearch", C.c_int32), ("max_fun", C.c_int32), ("consistent_gradient", C.c_int32),
        ("dt", C.c_double), ("mass", C.c_double), ("gravity", C.c_double),
        ("pos_bound", C.c_double), ("max_velocity", C.c_double), ("tilt_thrust", C.c_double),
        ("min_thrust", C.c_double), ("max_thrust", C.c_double),
        ("w_pos", C.c_double), ("w_vel", C.c_double), ("w_acc", C.c_double),
        ("w_thrust", C.c_double), ("gtol", C.c_double), ("ftol", C.c_double),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("f", C.c_double), ("nit", C.c_int32), ("nfev", C.c_int32), ("status", C.c_int32),
        ("task", C.c_int32), ("nseg_total", C.c_int32), ("nupdates", C.c_int32),
        ("nskip", C.c_int32), ("col_final", C.c_int32), ("nrestart", C.c_int32),
        ("pad_", C.c_int32), ("flops", C.c_double),
    ]


class Grid(C.Structure):
    _fields_ = [
        ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32),
        ("ox", C.c_int32), ("oy", C.c_int32), ("oz", C.c_int32),
        ("resolution", C.c_double), ("prior", C.c_double), ("occ", C.POINTER(C.c_float)),
        ("occ64", C.POINTER(C.c_double)),
    ]


FG_FN = C.CFUNCTYPE(C.c_double, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p)

_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        dp, ip, u8p = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
        L.orc_lbfgsb.argtypes = [C.c_int, C.c_int, dp, dp, dp, ip, FG_FN, C.c_void_p, C.c_double,
                                 C.c_double, C.c_int, C.c_int, C.c_int, C.POINTER(Stats)]
        L.orc_lbfgsb.restype = C.c_int
        L.orc_solve_batch.argtypes = [C.POINTER(Params), C.c_int64, dp, dp, dp, u8p, dp, dp, dp, ip,
                                      ip, ip, ip, dp, dp, dp, dp, dp, C.c_int]
        L.orc_solve_batch.restype = C.c_int
        L.orc_cold_start.argtypes = [C.POINTER(Params), dp, dp, dp, dp]
        L.orc_warm_start.argtypes = [C.POINTER(Params), dp, dp, dp, dp]
        L.orc_objective.argtypes = [C.POINTER(Params), dp, dp]
        L.orc_objective.restype = C.c_double
        L.orc_gradient.argtypes = [C.POINTER(Params), dp, dp, dp]
        L.orc_extract.argtypes = [C.POINTER(Params), dp, dp, dp, dp, dp]
        L.orc_query.argtypes = [C.POINTER(Grid), dp]
        L.orc_query.restype = C.c_double
        L.orc_traj_safe.argtypes = [C.POINTER(Grid), dp, C.c_int, C.c_double, C.c_double]
        L.orc_traj_safe.restype = C.c_int
        L.orc_trace_ray.argtypes = [C.c_double, dp, dp, C.c_double, ip, C.c_int]
        L.orc_trace_ray.restype = C.c_int
        L.orc_add_sphere.argtypes = [C.POINTER(Grid), dp, C.c_double, C.c_float]
        L.orc_add_sphere.restype = C.c_int
        L.orc_bayes.argtypes = [C.c_double, C.c_int]
        L.orc_bayes.restype = C.c_double
        L.orc_world_to_voxel.argtypes = [C.c_double, dp, ip]
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32)) if a is not None else None


def make_params(horizon=6, dt=0.0025, mass=1.5, gravity=9.81, max_velocity=10.0, max_thrust=25.0,
                min_thrust=2.0, max_tilt_angle=np.pi / 4, position_weight=100.0,
                velocity_weight=10.0, acceleration_weight=1.0, thrust_weight=0.1,
                max_iterations=15, convergence_tolerance=5e-2, max_corrections=10,
                max_linesearch=20, max_fun=15000, consistent_gradient=0, pos_bound=100.0) -> Params:
    """Defaults = SE3MPCConfig defaults (se3_mpc_planner.py:36-79) with the effective dt."""
    p = Params()
    p.horizon = int(horizon)
    p.max_iterations = int(max_iterations)
    p.max_corrections = int(max_corrections)
    p.max_linesearch = int(max_linesearch)
    p.max_fun = int(max_fun)
    p.consistent_gradient = int(consistent_gradient)
    p.dt, p.mass, p.gravity = float(dt), float(mass), float(gravity)
    p.pos_bound = float(pos_bound)
    p.max_velocity = float(max_velocity)
    p.tilt_thrust = float(max_thrust * np.sin(max_tilt_angle))
    p.min_thrust, p.max_thrust = float(min_thrust), float(max_thrust)
    p.w_pos, p.w_vel = float(position_weight), float(velocity_weight)
    p.w_acc, p.w_thrust = float(acceleration_weight), float(thrust_weight)
    p.gtol = float(convergence_tolerance)
    p.ftol = float(convergence_tolerance * 10)
    return p


@dataclass
class BatchResult:
    x: np.ndarray
    cost: np.ndarray
    nit: np.ndarray
    nfev: np.ndarray
    status: np.ndarray
    task: np.ndarray
    accelerations: np.ndarray
    attitudes: np.ndarray
    body_rates: np.ndarray
    thrusts: np.ndarray
    flops: float

    @property
    def positions(self):
        N = self.x.shape[1] // 9
        return self.x[:, : 3 * N].reshape(-1, N, 3)

    @property
    def velocities(self):
        N = self.x.shape[1] // 9
        return self.x[:, 3 * N: 6 * N].reshape(-1, N, 3)

    @property
    def thrust_vectors(self):
        N = self.x.shape[1] // 9
        return self.x[:, 6 * N:].reshape(-1, N, 3)


def solve_batch(p: Params, p0, v0, goal, has_goal=None, x_warm=None, nthreads=1, grid=None,
                obstacle_weight=0.0, free_level=0.5) -> BatchResult:
    """grid: DenseGrid -> adds the occupancy-grid obstacle penalty (extension, self-oracle)."""
    p0 = np.ascontiguousarray(p0, dtype=np.float64).reshape(-1, 3)
    B = p0.shape[0]
    v0 = np.ascontiguousarray(v0, dtype=np.float64).reshape(B, 3)
    goal = np.ascontiguousarray(goal, dtype=np.float64).reshape(B, 3)
    N = p.horizon
    n = 9 * N
    hg = None
    if has_goal is not None:
        hg = np.ascontiguousarray(has_goal, dtype=np.uint8).reshape(B)
    xw = None
    if x_warm is not None:
        xw = np.ascontiguousarray(x_warm, dtype=np.float64).reshape(B, n)
    x = np.zeros((B, n))
    cost = np.zeros(B)
    nit = np.zeros(B, np.int32)
    nfev = np.zeros(B, np.int32)
    status = np.zeros(B, np.int32)
    task = np.zeros(B, np.int32)
    acc = np.zeros((B, N, 3))
    att = np.zeros((B, N, 3))
    rates = np.zeros((B, N, 3))
    thrust = np.zeros((B, N))
    fl = C.c_double(0.0)
    L = lib()
    L.orc_solve_batch_grid.restype = C.c_int
    rc = L.orc_solve_batch_grid(
        C.byref(p), C.c_int64(B), _dp(p0), _dp(v0), _dp(goal),
        hg.ctypes.data_as(C.POINTER(C.c_uint8)) if hg is not None else None, _dp(xw), _dp(x),
        _dp(cost), _ip(nit), _ip(nfev), _ip(status), _ip(task), _dp(acc), _dp(att), _dp(rates),
        _dp(thrust), C.byref(fl), C.c_int(int(nthreads)),
        C.byref(grid.g) if grid is not None else None, C.c_double(float(obstacle_weight)),
        C.c_double(float(free_level)))
    if rc != 0:
        raise RuntimeError(f"orc_solve_batch failed: {rc}")
    return BatchResult(x, cost, nit, nfev, status, task, acc, att, rates, thrust, fl.value)


def lbfgsb(fun_and_grad, x0, lo, hi, nbd, m=10, factr=1e7, pgtol=1e-5, maxiter=15000,
           maxfun=15000, maxls=20, trace=None):
    """Generic oracle L-BFGS-B with a Python f/g callback (for validation against SciPy)."""
    x = np.array(x0, dtype=np.float64).copy()
    n = x.size
    lo = np.ascontiguousarray(lo, dtype=np.float64)
    hi = np.ascontiguousarray(hi, dtype=np.float64)
    nbd = np.ascontiguousarray(nbd, dtype=np.int32)

    def _cb(nn, xp, gp, _user):
        xv = np.ctypeslib.as_array(xp, shape=(nn,))
        gv = np.ctypeslib.as_array(gp, shape=(nn,))
        f, g = fun_and_grad(xv.copy())
        gv[:] = g
        if trace is not None:
            trace.append((xv.copy(), float(f)))
        return float(f)

    st = Stats()
    rc = lib().orc_lbfgsb(n, m, _dp(x), _dp(lo), _dp(hi), _ip(nbd), FG_FN(_cb), None, factr, pgtol,
                          maxiter, maxfun, maxls, C.byref(st))
    if rc != 0:
        raise RuntimeError("orc_lbfgsb failed")
    return x, st


def extract(p: Params, x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    N = p.horizon
    acc, att, rates, thrust = np.zeros((N, 3)), np.zeros((N, 3)), np.zeros((N, 3)), np.zeros(N)
    lib().orc_extract(C.byref(p), _dp(x), _dp(acc), _dp(att), _dp(rates), _dp(thrust))
    return acc, att, rates, thrust


def cold_start(p: Params, p0, v0, goal):
    x0 = np.zeros(9 * p.horizon)
    p0 = np.ascontiguousarray(p0, dtype=np.float64)
    v0 = np.ascontiguousarray(v0, dtype=np.float64)
    g = None if goal is None else np.ascontiguousarray(goal, dtype=np.float64)
    lib().orc_cold_start(C.byref(p), _dp(p0), _dp(v0), _dp(g), _dp(x0))
    return x0


def warm_start(p: Params, p0, v0, prev_x):
    x0 = np.zeros(9 * p.horizon)
    p0 = np.ascontiguousarray(p0, dtype=np.float64)
    v0 = np.ascontiguousarray(v0, dtype=np.float64)
    px = np.ascontiguousarray(prev_x, dtype=np.float64)
    lib().orc_warm_start(C.byref(p), _dp(p0), _dp(v0), _dp(px), _dp(x0))
    return x0


def objective(p: Params, x, goal):
    x = np.ascontiguousarray(x, dtype=np.float64)
    g = None if goal is None else np.ascontiguousarray(goal, dtype=np.float64)
    return lib().orc_objective(C.byref(p), _dp(x), _dp(g))


def gradient(p: Params, x, goal):
    x = np.ascontiguousarray(x, dtype=np.float64)
    g = None if goal is None else np.ascontiguousarray(goal, dtype=np.float64)
    out = np.zeros_like(x)
    lib().orc_gradient(C.byref(p), _dp(x), _dp(g), _dp(out))
    return out


class DenseGrid:
    """Dense occupancy grid standing in for the reference's sparse dict (mapper :77-78)."""

    def __init__(self, shape=(256, 256, 256), origin_voxel=(-128, -128, -128), resolution=0.2,
                 prior=0.5):
        nx, ny, nz = shape
        self.occ = np.full((nz, ny, nx), prior, dtype=np.float32)
        self.g = Grid(nx, ny, nz, origin_voxel[0], origin_voxel[1], origin_voxel[2],
                      float(resolution), float(prior),
                      self.occ.ctypes.data_as(C.POINTER(C.c_float)))

    @classmethod
    def from_cells(cls, occ, origin_voxel, resolution, prior):
        """A grid over the given (nz, ny, nx) cells, float32 or float64 (the penalty reads float64
        cells as stored; the mapper queries read only float32 grids)."""
        occ = np.ascontiguousarray(occ)
        assert occ.ndim == 3 and occ.dtype in (np.float32, np.float64)
        nz, ny, nx = occ.shape
        self = cls.__new__(cls)
        self.occ = occ
        f32 = occ if occ.dtype == np.float32 else None
        self.g = Grid(nx, ny, nz, origin_voxel[0], origin_voxel[1], origin_voxel[2], float(resolution),
                      float(prior), None if f32 is None else f32.ctypes.data_as(C.POINTER(C.c_float)),
                      None if f32 is not None else occ.ctypes.data_as(C.POINTER(C.c_double)))
        return self

    def _mapper_grid(self):
        """The grid the mapper queries read: they take float32 cells only."""
        if not self.g.occ:
            raise TypeError("the mapper queries read float32 cells; this grid holds float64 cells")
        return self.g

    def add_sphere(self, center, radius, value=0.9):
        self._mapper_grid()
        c = np.ascontiguousarray(center, dtype=np.float64)
        return lib().orc_add_sphere(C.byref(self.g), _dp(c), float(radius), float(value))

    def query(self, pos):
        pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 3)
        g = self._mapper_grid()
        return np.array([lib().orc_query(C.byref(g), _dp(q)) for q in pos])

    def penalty(self, pos, weight, free_level=0.5):
        """(f, grad[3]) of the obstacle penalty at one position (orc_grid_penalty)."""
        L = lib()
        L.orc_grid_penalty.restype = C.c_double
        q = np.ascontiguousarray(pos, dtype=np.float64).reshape(3)
        g = np.zeros(3)
        f = L.orc_grid_penalty(C.byref(self.g), C.c_double(float(weight)), C.c_double(float(free_level)),
                               _dp(q), _dp(g))
        return f, g

    def traj_safe(self, positions, margin, threshold):
        q = np.ascontiguousarray(positions, dtype=np.float64).reshape(-1, 3)
        return lib().orc_traj_safe(C.byref(self._mapper_grid()), _dp(q), q.shape[0], float(margin),
                                   float(threshold))


def update_map(grid: "DenseGrid", occ64, pos, direction, hit, obs_max_range, mapper_max_range, counts=None):
    """Sequential update_map on a double-precision copy of the grid (modified in place)."""
    L = lib()
    L.orc_update_map.restype = C.c_int64
    pos = np.ascontiguousarray(pos, np.float64).reshape(-1, 3)
    n = len(pos)
    d = np.ascontiguousarray(direction, np.float64).reshape(n, 3)
    h = np.ascontiguousarray(hit, np.float64).reshape(n)
    mr = np.ascontiguousarray(obs_max_range, np.float64).reshape(n)
    assert occ64.dtype == np.float64 and occ64.flags.c_contiguous and occ64.shape == grid.occ.shape
    return L.orc_update_map(C.byref(grid._mapper_grid()), _dp(occ64), _ip(counts) if counts is not None else None,
                            C.c_int64(n), _dp(pos), _dp(d), _dp(h), _dp(mr), C.c_double(float(mapper_max_range)))


def trace_ray(res, start, direction, distance, max_vox=4096):
    s = np.ascontiguousarray(start, dtype=np.float64)
    d = np.ascontiguousarray(direction, dtype=np.float64)
    out = np.zeros((max_vox, 3), np.int32)
    n = lib().orc_trace_ray(float(res), _dp(s), _dp(d), float(distance), _ip(out), max_vox)
    return out[: min(n, max_vox)].copy(), n


def bayes(p, hit):
    return lib().orc_bayes(float(p), int(bool(hit)))
