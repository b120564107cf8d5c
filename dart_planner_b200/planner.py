"""Host side of the B200 SE(3)-MPC path.

* ``SE3MPCPlanner`` -- drop-in for the reference class
  (src/dart_planner/planning/se3_mpc_planner.py:82-757): same constructor, methods, dict keys
  and ``Trajectory`` fields; one problem per call, solved on the GPU through the C ABI.
* ``plan_batch`` / ``BatchWorkspace`` -- the new batched entry point: thousands of independent
  problems (Monte-Carlo initial states, candidate goals, multi-start warm starts) per call.

PyTorch is used only for device memory, pinned host memory and streams.
"""
from __future__ import annotations

import ctypes as C
import logging
import os
import time
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _cabi
from .config import (AttrDict, REFERENCE_CONTROL_FREQUENCY_HZ, SE3MPCConfig, load_planner_config,
                     make_params, to_si)
from .types import DroneState, Trajectory

logger = logging.getLogger(__name__)


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("dart_planner_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch


def _ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


# row layout of the fp64 output block: [x 9N | cost 1 | acc 3N | att 3N | rates 3N | thrust N]
def out_rows(N: int) -> int:
    return 19 * N + 1


@dataclass
class BatchSolution:
    """Result of a batched solve.  Device tensors in batch-major SoA; the properties give the
    reference's (B, N, 3) views without copying."""

    N: int
    B: int
    out: Any     # (19N+1, ld) float64
    meta: Any    # (4, ld) int32 rows: nit, nfev, status, task
    hit: Any = None   # (ld,) int32 first colliding position index (-1 safe) when a map was given

    def _rows(self, lo, hi):
        return self.out[lo:hi, : self.B]

    def _bn3(self, lo):
        return self._rows(lo, lo + 3 * self.N).t().view(self.B, self.N, 3)

    @property
    def x(self):  # (B, 9N) in the reference's packed order
        return self._rows(0, 9 * self.N).t()

    @property
    def positions(self):
        return self._bn3(0)

    @property
    def velocities(self):
        return self._bn3(3 * self.N)

    @property
    def thrust_vectors(self):
        return self._bn3(6 * self.N)

    @property
    def cost(self):
        return self.out[9 * self.N, : self.B]

    @property
    def accelerations(self):
        return self._bn3(9 * self.N + 1)

    @property
    def attitudes(self):
        return self._bn3(12 * self.N + 1)

    @property
    def body_rates(self):
        return self._bn3(15 * self.N + 1)

    @property
    def thrusts(self):
        return self._rows(18 * self.N + 1, 19 * self.N + 1).t()

    @property
    def nit(self):
        return self.meta[0, : self.B]

    @property
    def nfev(self):
        return self.meta[1, : self.B]

    @property
    def status(self):
        return self.meta[2, : self.B]

    @property
    def task(self):
        return self.meta[3, : self.B]

    @property
    def success(self):
        return self.status == 0

    @property
    def first_hit(self):
        """is_trajectory_safe's collision index per problem (-1 = safe); needs `grid=`."""
        if self.hit is None:
            raise ValueError("no occupancy grid was passed to the solve")
        return self.hit[: self.B]

    @property
    def safe(self):
        return self.first_hit < 0

    def numpy(self) -> "HostSolution":
        """Copy everything to host ndarrays with the reference's shapes.  The SoA block is
        transposed on the device (one pass over HBM instead of seven strided NumPy transposes on
        the host); the result's fields are views of one (B, 19N+1) host array, like the
        reference's views into ``result.x``."""
        out_t = self.out[:, : self.B].t().contiguous().cpu().numpy()
        meta = self.meta[:, : self.B].cpu().numpy()
        hs = HostSolution.from_rows(self.N, out_t, meta)
        if self.hit is not None:
            hs.first_hit = self.hit[: self.B].cpu().numpy()
        return hs


@dataclass
class ControlsSolution:
    """What a controls row carries: the thrust commands of every problem and the solver's report."""
    thrust_vectors: np.ndarray
    cost: np.ndarray
    nit: np.ndarray
    nfev: np.ndarray
    status: np.ndarray
    task: np.ndarray

    @property
    def success(self):
        return self.status == 0


_DERIVED = ("accelerations", "attitudes", "body_rates", "thrusts")


@dataclass
class HostSolution:
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
    first_hit: Optional[np.ndarray] = None

    def __getattr__(self, name):
        # solution rows (from_solution_rows): the derived arrays are not transferred; they are
        # evaluated from the thrust rows of x on first access (derive.py, :582-654)
        if name in _DERIVED and "_derive_with" in self.__dict__:
            from .derive import derive_from_thrust
            dt, mass, gravity = self.__dict__["_derive_with"]
            vals = derive_from_thrust(self.thrust_vectors, dt, mass, gravity)
            for k, v in zip(_DERIVED, vals):
                self.__dict__[k] = v
            return self.__dict__[name]
        raise AttributeError(name)

    @staticmethod
    def from_blocks(N: int, out: np.ndarray, meta: np.ndarray) -> "HostSolution":
        B = out.shape[1]

        def bn3(lo):
            return np.ascontiguousarray(out[lo:lo + 3 * N].T).reshape(B, N, 3)

        return HostSolution(
            x=np.ascontiguousarray(out[: 9 * N].T), cost=out[9 * N].copy(), nit=meta[0].copy(),
            nfev=meta[1].copy(), status=meta[2].copy(), task=meta[3].copy(),
            accelerations=bn3(9 * N + 1), attitudes=bn3(12 * N + 1), body_rates=bn3(15 * N + 1),
            thrusts=np.ascontiguousarray(out[18 * N + 1: 19 * N + 1].T))

    @staticmethod
    def from_rows(N: int, rows: np.ndarray, meta: np.ndarray) -> "HostSolution":
        """rows: (B, 19N+1) problem-major array [x 9N | cost | acc 3N | att 3N | rates 3N | thrust N]."""
        B = rows.shape[0]

        def bn3(lo):
            return rows[:, lo:lo + 3 * N].reshape(B, N, 3)

        return HostSolution(
            x=rows[:, : 9 * N], cost=rows[:, 9 * N], nit=meta[0], nfev=meta[1], status=meta[2],
            task=meta[3], accelerations=bn3(9 * N + 1), attitudes=bn3(12 * N + 1),
            body_rates=bn3(15 * N + 1), thrusts=rows[:, 18 * N + 1: 19 * N + 1])

    @staticmethod
    def from_packed_rows(N: int, rows: np.ndarray) -> "HostSolution":
        """rows: (B, stride) float64 result rows of `dart_se3mpc_solve_batch_rows` (layout in
        include/dart_se3mpc.h): views, no copies."""
        meta = rows[:, 19 * N + 1: 19 * N + 4].view(np.int32)         # (B, 6)
        sol = HostSolution.from_rows(N, rows, meta.T)
        sol.first_hit = None if (meta[:, 4] == -2).all() else meta[:, 4]
        return sol

    @staticmethod
    def from_solution_rows(N: int, rows: np.ndarray, params) -> "HostSolution":
        """rows: (B, stride) solution rows (DART_ROWS_SOLUTION: x | cost | counters): views, no
        copies.  accelerations / attitudes / body_rates / thrusts are derived on first access."""
        meta = rows[:, 9 * N + 1: 9 * N + 4].view(np.int32)           # (B, 6)
        sol = HostSolution(x=rows[:, : 9 * N], cost=rows[:, 9 * N], nit=meta[:, 0], nfev=meta[:, 1],
                           status=meta[:, 2], task=meta[:, 3], accelerations=None, attitudes=None,
                           body_rates=None, thrusts=None)
        for k in _DERIVED:
            del sol.__dict__[k]
        sol.__dict__["_derive_with"] = (float(params.dt), float(params.mass), float(params.gravity))
        sol.first_hit = None if (meta[:, 4] == -2).all() else meta[:, 4]
        return sol

    @staticmethod
    def from_control_rows(N: int, rows: np.ndarray) -> "ControlsSolution":
        """rows: (B, stride) controls rows (DART_ROWS_CONTROLS): views, no copies."""
        meta = rows[:, 3 * N + 1: 3 * N + 4].view(np.int32)
        return ControlsSolution(thrust_vectors=rows[:, : 3 * N].reshape(-1, N, 3), cost=rows[:, 3 * N],
                                nit=meta[:, 0], nfev=meta[:, 1], status=meta[:, 2], task=meta[:, 3])

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

    @property
    def success(self):
        return self.status == 0


def sphere_rows(spheres) -> np.ndarray:
    """(centers (S, 3), radii (S,)) from NumPy or torch -> the (S, 4) float64 list [cx cy cz r] of
    ``dart_spheres``."""
    centers, radii = spheres
    to_np = lambda a: a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)  # noqa: E731
    c = np.asarray(to_np(centers), np.float64).reshape(-1, 3)
    r = np.asarray(to_np(radii), np.float64).reshape(-1)
    if len(r) != len(c):
        raise ValueError("spheres: centers (S, 3) and radii (S,) must have the same length")
    return np.ascontiguousarray(np.concatenate([c, r[:, None]], axis=1))


def reference_rows(P, V, B: int, ld: int, device):
    """(P (B, T, 3), V (B, T, 3) or None) from NumPy or torch -> the (6T, ld) float64 device block of
    ``dart_track_ref`` (rows 3j+c position, 3T+3j+c velocity of sample j; V None = zero velocities)."""
    torch = _torch()
    as_t = lambda a: (a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, np.float64))).to(  # noqa: E731
        device, torch.float64)
    Pt = as_t(P)
    if Pt.dim() != 3 or Pt.shape[0] != B or Pt.shape[2] != 3 or Pt.shape[1] < 1:
        raise ValueError(f"reference positions must be (B={B}, T, 3), got {tuple(Pt.shape)}")
    T = Pt.shape[1]
    Vt = torch.zeros_like(Pt) if V is None else as_t(V)
    if tuple(Vt.shape) != tuple(Pt.shape):
        raise ValueError(f"reference velocities must be (B, T, 3) like the positions, got {tuple(Vt.shape)}")
    rows = torch.zeros((6 * T, ld), dtype=torch.float64, device=device)
    rows[: 3 * T, :B] = Pt.reshape(B, 3 * T).t()
    rows[3 * T:, :B] = Vt.reshape(B, 3 * T).t()
    return rows


def solve_batch_tensors(params: _cabi.Params, inp, B: int, *, has_goal=None, x_warm=None,
                        warm_mask=None, out=None, meta=None, stream=None,
                        outputs: str = "all", grid=None, safety_margin: float = 1.0,
                        collision_threshold: float = 0.6, hit=None, penalty_grid=None,
                        spheres: Optional[_cabi.Spheres] = None,
                        reference: Optional[_cabi.TrackRef] = None) -> BatchSolution:
    """Lowest Python level: device tensors in, device tensors out, one kernel launch.

    inp      : (9, ld) float64 CUDA tensor, rows [p0 xyz | v0 xyz | goal xyz]
    has_goal : (ld,) uint8 or None;  x_warm : (9N, ld) float64 or None;  warm_mask (ld,) uint8
    out/meta : optional preallocated (19N+1, ld) float64 / (4, ld) int32
    outputs  : "all" | "controls" (x, cost, counters only; no derived rows are written)
    grid     : DenseOccupancyGrid or None; when given, the kernel also runs the reference's
               post-hoc `is_trajectory_safe(positions, safety_margin, collision_threshold)` on
               every solved trajectory (fused, same launch) -> BatchSolution.first_hit
    penalty_grid : DenseOccupancyGrid or None; the grid the obstacle penalty (gradient_mode 2 / 4)
               reads instead of ``grid``.  ``grid`` is then only the safety check's, which runs as
               a second launch (dart_map_traj_safe_batch, the same test as the fused check) on
               the solved positions
    spheres  : _cabi.Spheres over a device list, or None; the sphere penalty of gradient_mode 5 / 6
               (``grid`` then serves only the fused safety check)
    reference : _cabi.TrackRef over a (6T, ld) device block, or None; the per-timestep reference of
               gradient_mode 7 / 8 (``inp``'s goal rows are not read)
    """
    torch = _torch()
    L = _cabi.lib()
    N = int(params.horizon)
    ld = inp.shape[1]
    assert inp.dtype == torch.float64 and inp.is_cuda and inp.shape[0] == 9 and inp.is_contiguous()
    assert 0 <= B <= ld
    if out is None:
        # rows the kernel does not write (outputs != "all") must not read as garbage
        alloc = torch.empty if outputs == "all" else torch.zeros
        out = alloc((out_rows(N), ld), dtype=torch.float64, device=inp.device)
    if meta is None:
        meta = torch.empty((4, ld), dtype=torch.int32, device=inp.device)
    assert out.shape == (out_rows(N), ld) and out.is_contiguous() and out.dtype == torch.float64
    assert meta.shape == (4, ld) and meta.is_contiguous() and meta.dtype == torch.int32
    for t, rows, dt in ((has_goal, None, torch.uint8), (warm_mask, None, torch.uint8),
                        (x_warm, 9 * N, torch.float64)):
        if t is not None:
            assert t.is_cuda and t.is_contiguous() and t.dtype == dt and t.shape[-1] == ld
            assert rows is None or t.shape[0] == rows
    if stream is None:
        stream = torch.cuda.current_stream(inp.device)
    base, es = out.data_ptr(), 8 * ld
    derived = outputs == "all"
    g = None
    if grid is not None:
        g = grid._grid()
        if hit is None:
            hit = torch.empty(ld, dtype=torch.int32, device=inp.device)
        assert hit.is_cuda and hit.dtype == torch.int32 and hit.shape == (ld,) and hit.is_contiguous()
    fused = g is not None and penalty_grid is None
    if penalty_grid is not None:
        g = penalty_grid._grid()
    args = (C.byref(params), B, ld, inp.data_ptr(), inp.data_ptr() + 3 * es, inp.data_ptr() + 6 * es,
            _ptr(has_goal), _ptr(x_warm), _ptr(warm_mask),
            base, base + 9 * N * es,
            meta.data_ptr(), meta.data_ptr() + 4 * ld, meta.data_ptr() + 8 * ld, meta.data_ptr() + 12 * ld,
            base + (9 * N + 1) * es if derived else None,
            base + (12 * N + 1) * es if derived else None,
            base + (15 * N + 1) * es if derived else None,
            base + (18 * N + 1) * es if derived else None)
    check = (C.byref(g) if g is not None else None, float(safety_margin), float(collision_threshold),
             hit.data_ptr() if fused else None, stream.cuda_stream)
    with torch.cuda.device(inp.device):
        if reference is not None:
            name = "dart_se3mpc_solve_batch_track"
            rc = L.dart_se3mpc_solve_batch_track(*args[:5], *args[6:], C.byref(reference),
                                                 None if spheres is None else C.byref(spheres), *check)
        elif spheres is None:
            name = "dart_se3mpc_solve_batch_map"
            rc = L.dart_se3mpc_solve_batch_map(*args, *check)
        else:
            name = "dart_se3mpc_solve_batch_spheres"
            rc = L.dart_se3mpc_solve_batch_spheres(*args, C.byref(spheres), *check)
    _cabi.check(rc, name)
    if grid is not None and not fused:
        grid.trajectories_safe_soa(out[: 3 * N], B, N, safety_margin, collision_threshold, out=hit, stream=stream)
    return BatchSolution(N=N, B=B, out=out, meta=meta, hit=hit if grid is not None else None)


class BatchWorkspace:
    """Preallocated device (and pinned host) buffers for repeated batched solves of one shape.

    ``solve_device()`` launches on resident inputs; ``solve_host(p0, v0, goal)`` is the
    end-to-end call: pinned H2D copy of the inputs, one launch, D2H copy of the full result.
    """

    def __init__(self, params: _cabi.Params, B: int, device=None, pinned: bool = True,
                 outputs: str = "all"):
        torch = _torch()
        self.params = params
        self.N = int(params.horizon)
        self.B = int(B)
        self.ld = max(32, (self.B + 31) // 32 * 32)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.outputs = outputs
        self.inp = torch.zeros((9, self.ld), dtype=torch.float64, device=self.device)
        self.out = torch.zeros((out_rows(self.N), self.ld), dtype=torch.float64, device=self.device)
        self.meta = torch.zeros((4, self.ld), dtype=torch.int32, device=self.device)
        self.has_goal = None
        self.x_warm = None
        self.warm_mask = None
        self.grid, self.safety_margin, self.collision_threshold, self.hit = None, 1.0, 0.6, None
        self.penalty_grid = None
        self.spheres = self.spheres_dev = None
        self.reference = self.reference_dev = None
        self.h_inp = self.h_out = self.h_meta = self.h_rows = None
        # DART_ROWS_FULL / DART_ROWS_CONTROLS / DART_ROWS_SOLUTION
        if outputs not in ("all", "controls", "solution"):
            raise ValueError("outputs must be 'all', 'controls' or 'solution'")
        self.row_kind = {"all": 0, "controls": 1, "solution": 2}[outputs]
        self.row_stride = int(_cabi.lib().dart_se3mpc_row_stride(C.byref(params), self.row_kind))
        if pinned:
            self.h_inp = torch.zeros((9, self.ld), dtype=torch.float64).pin_memory()
            self.h_out = torch.zeros((out_rows(self.N), self.ld), dtype=torch.float64).pin_memory()
            self.h_meta = torch.zeros((4, self.ld), dtype=torch.int32).pin_memory()

    @property
    def h2d_bytes(self) -> int:
        return 9 * self.B * 8

    @property
    def d2h_bytes(self) -> int:
        rows = out_rows(self.N) if self.outputs == "all" else 9 * self.N + 1
        return rows * self.B * 8 + 4 * self.B * 4

    def set_inputs_device(self, p0, v0, goal):
        """(B,3) tensors/arrays -> resident SoA input block (not part of any timed region)."""
        torch = _torch()
        for i, a in enumerate((p0, v0, goal)):
            t = torch.as_tensor(np.asarray(a, dtype=np.float64) if not torch.is_tensor(a) else a,
                                dtype=torch.float64).to(self.device)
            self.inp[3 * i: 3 * i + 3, : self.B] = t.reshape(self.B, 3).t()

    def set_warm(self, x_prev, mask=None):
        """x_prev: (B, 9N) previous solutions (reference packed order) or a (9N, ld) SoA tensor."""
        torch = _torch()
        if x_prev is None:
            self.x_warm = self.warm_mask = None
            return
        if torch.is_tensor(x_prev) and x_prev.is_cuda and tuple(x_prev.shape) == (9 * self.N, self.ld):
            self.x_warm = x_prev
        else:
            xp = torch.as_tensor(np.asarray(x_prev, np.float64) if not torch.is_tensor(x_prev) else x_prev,
                                 dtype=torch.float64).to(self.device).reshape(self.B, 9 * self.N)
            if self.x_warm is None or tuple(self.x_warm.shape) != (9 * self.N, self.ld):
                self.x_warm = torch.zeros((9 * self.N, self.ld), dtype=torch.float64, device=self.device)
            self.x_warm[:, : self.B] = xp.t()
        if mask is not None:
            m = torch.as_tensor(np.asarray(mask, np.uint8) if not torch.is_tensor(mask) else mask).to(
                self.device, torch.uint8).reshape(self.B)
            self.warm_mask = torch.zeros(self.ld, dtype=torch.uint8, device=self.device)
            self.warm_mask[: self.B] = m
        else:
            self.warm_mask = None

    def set_has_goal(self, has_goal):
        torch = _torch()
        if has_goal is None:
            self.has_goal = None
            return
        h = torch.as_tensor(np.asarray(has_goal, np.uint8)).to(self.device, torch.uint8).reshape(self.B)
        self.has_goal = torch.ones(self.ld, dtype=torch.uint8, device=self.device)
        self.has_goal[: self.B] = h

    def set_map(self, grid, safety_margin: float = 1.0, collision_threshold: float = 0.6, penalty_grid=None):
        """Attach a DenseOccupancyGrid: every solve also runs the fused trajectory safety check.
        ``penalty_grid``: a separate grid for the obstacle penalty (see solve_batch_tensors; SoA
        solves only)."""
        torch = _torch()
        self.grid, self.safety_margin, self.collision_threshold = grid, safety_margin, collision_threshold
        self.penalty_grid = penalty_grid
        self.hit = None if grid is None else torch.full((self.ld,), -1, dtype=torch.int32, device=self.device)

    def set_spheres(self, spheres, margin: float = 0.0):
        """The sphere list of the obstacle penalty (gradient_mode 5 / 6): (centers (S, 3), radii (S,)),
        every radius inflated by ``margin``; uploaded once, used by every SoA solve.  None removes it."""
        torch = _torch()
        if spheres is None:
            self.spheres = self.spheres_dev = None
            return
        rows = sphere_rows(spheres)
        self.spheres_dev = torch.as_tensor(rows).to(self.device) if len(rows) else None
        self.spheres = _cabi.Spheres(len(rows), 0, _ptr(self.spheres_dev), float(margin))

    def set_reference(self, P, V=None, start: int = 0):
        """The per-timestep reference of gradient_mode 7 / 8: positions P (B, T, 3) and velocities V
        (B, T, 3) or None (zero), NumPy or torch; timestep k of every solve tracks sample
        min(start + k, T - 1).  Uploaded once, used by every SoA solve.  P None removes it."""
        if P is None:
            self.reference = self.reference_dev = None
            return
        if int(start) < 0:
            raise ValueError("reference start must be >= 0")
        self.reference_dev = reference_rows(P, V, self.B, self.ld, self.device)
        self.reference = _cabi.TrackRef(self.reference_dev.shape[0] // 6, int(start), self.reference_dev.data_ptr())

    def solve_device(self, stream=None) -> BatchSolution:
        return solve_batch_tensors(self.params, self.inp, self.B, has_goal=self.has_goal,
                                   x_warm=self.x_warm, warm_mask=self.warm_mask, out=self.out,
                                   meta=self.meta, stream=stream, outputs=self.outputs,
                                   grid=self.grid, safety_margin=self.safety_margin,
                                   collision_threshold=self.collision_threshold, hit=self.hit,
                                   penalty_grid=self.penalty_grid, spheres=self.spheres,
                                   reference=self.reference)

    def stage_host_inputs(self, p0, v0, goal):
        """Write (B,3) host arrays into the pinned SoA staging block (host-side transpose)."""
        h = self.h_inp.numpy()
        h[0:3, : self.B] = np.asarray(p0, np.float64).reshape(self.B, 3).T
        h[3:6, : self.B] = np.asarray(v0, np.float64).reshape(self.B, 3).T
        h[6:9, : self.B] = np.asarray(goal, np.float64).reshape(self.B, 3).T

    def solve_staged(self, stream=None):
        """pinned H2D -> solve -> pinned D2H, all on one stream; returns after synchronising."""
        torch = _torch()
        if (self.B >= 65536 and self.B == self.ld and self.has_goal is None and self.x_warm is None
                and self.grid is None and self.spheres is None and self.reference is None):
            return self._solve_staged_pipelined()
        stream = stream or torch.cuda.current_stream(self.device)
        with torch.cuda.stream(stream):
            self.inp.copy_(self.h_inp, non_blocking=True)
            self.solve_device(stream)
            nrows = out_rows(self.N) if self.outputs == "all" else 9 * self.N + 1
            self.h_out[:nrows].copy_(self.out[:nrows], non_blocking=True)
            self.h_meta.copy_(self.meta, non_blocking=True)
        stream.synchronize()
        return self.h_out, self.h_meta

    @property
    def rows_supported(self) -> bool:
        """Row output: no entry of it takes a sphere list or a reference."""
        return (self.row_stride > 0 and self.h_inp is not None and self.spheres is None
                and self.reference is None)

    @property
    def d2h_bytes_rows(self) -> int:
        return self.row_stride * 8 * self.B

    def solve_rows(self, stream=None, wait: bool = True):
        """Zero-copy end-to-end solve: ONE launch whose kernel reads the pinned input block and
        writes every problem's result row straight into pinned host memory over PCIe (full
        128-byte lines); no copy in either direction.  Returns the pinned (B, stride) row block
        (`HostSolution.from_packed_rows(N, rows.numpy())` gives the named views).  A workspace
        built with ``outputs="solution"`` gets solution rows (x, cost, counters -- what
        ``scipy.optimize.minimize`` returns; `HostSolution.from_solution_rows` derives the rest on
        the host on first access), half the bytes; ``outputs="controls"`` gets controls rows:
        thrust vectors, cost and counters only (`HostSolution.from_control_rows`), a fifth."""
        torch = _torch()
        if self.penalty_grid is not None:
            raise ValueError("row output has no separate penalty grid")
        if self.spheres is not None:
            raise ValueError("row output has no sphere penalty")
        if self.reference is not None:
            raise ValueError("row output has no reference tracking")
        if not self.rows_supported:
            raise RuntimeError("row output needs pinned buffers and a horizon of at most 25 steps")
        if self.h_rows is None:
            self.h_rows = torch.zeros((self.ld, self.row_stride), dtype=torch.float64).pin_memory()
        stream = stream or torch.cuda.current_stream(self.device)
        es = 8 * self.ld
        hi = self.h_inp.data_ptr()
        g = self.grid._grid() if self.grid is not None else None
        with torch.cuda.device(self.device):
            rc = _cabi.lib().dart_se3mpc_solve_batch_rows(
                C.byref(self.params), self.B, self.ld, hi, hi + 3 * es, hi + 6 * es,
                _ptr(self.has_goal), _ptr(self.x_warm), _ptr(self.warm_mask),
                self.h_rows.data_ptr(), self.row_stride, self.row_kind,
                C.byref(g) if g is not None else None, float(self.safety_margin),
                float(self.collision_threshold), 1 if g is not None else 0, stream.cuda_stream)
        _cabi.check(rc, "dart_se3mpc_solve_batch_rows")
        if wait:
            stream.synchronize()
        return self.h_rows[: self.B]

    def solve_rows_device(self, stream=None, rows_ptr: Optional[int] = None):
        """Row output from the resident inputs into DEVICE memory (what `ShardedSolver` gathers:
        one contiguous row per problem, so a rank's slice is one contiguous block); returns the
        (B, stride) device tensor.  With ``rows_ptr`` the rows go to that address instead -- B rows
        of `row_stride` doubles, 128-byte aligned, device memory or page-locked mapped host memory
        (the shared block of `ShardedSolver(transport="host_block")`) -- and nothing is returned.
        Asynchronous."""
        torch = _torch()
        if self.penalty_grid is not None:
            raise ValueError("row output has no separate penalty grid")
        if self.spheres is not None:
            raise ValueError("row output has no sphere penalty")
        if self.reference is not None:
            raise ValueError("row output has no reference tracking")
        if self.row_stride <= 0:
            raise RuntimeError("row output needs a horizon of at most 25 steps (64 for controls rows)")
        if rows_ptr is None and getattr(self, "d_rows", None) is None:
            self.d_rows = torch.zeros((self.ld, self.row_stride), dtype=torch.float64, device=self.device)
        stream = stream or torch.cuda.current_stream(self.device)
        es = 8 * self.ld
        di = self.inp.data_ptr()
        g = self.grid._grid() if self.grid is not None else None
        with torch.cuda.device(self.device):
            rc = _cabi.lib().dart_se3mpc_solve_batch_rows(
                C.byref(self.params), self.B, self.ld, di, di + 3 * es, di + 6 * es,
                _ptr(self.has_goal), _ptr(self.x_warm), _ptr(self.warm_mask),
                rows_ptr if rows_ptr is not None else self.d_rows.data_ptr(), self.row_stride, self.row_kind,
                C.byref(g) if g is not None else None, float(self.safety_margin),
                float(self.collision_threshold), 1 if (g is not None and self.row_kind != 1) else 0,
                stream.cuda_stream)
        _cabi.check(rc, "dart_se3mpc_solve_batch_rows")
        return None if rows_ptr is not None else self.d_rows[: self.B]

    def _solve_staged_pipelined(self):
        """Large batches: the C host entry splits the batch into chunks on two streams so the
        read-back of one chunk overlaps the solve of the next (pinned buffers: fully async)."""
        N, es = self.N, 8 * self.ld
        hi, ho, hm = self.h_inp.data_ptr(), self.h_out.data_ptr(), self.h_meta.data_ptr()
        derived = self.outputs == "all"
        with _torch().cuda.device(self.device):
            rc = _cabi.lib().dart_se3mpc_solve_batch_host(
                C.byref(self.params), self.B, hi, hi + 3 * es, hi + 6 * es, None, None,
                ho, ho + 9 * N * es, hm, hm + 4 * self.ld, hm + 8 * self.ld,
                ho + (9 * N + 1) * es if derived else None, ho + (12 * N + 1) * es if derived else None,
                ho + (15 * N + 1) * es if derived else None, ho + (18 * N + 1) * es if derived else None)
        _cabi.check(rc, "dart_se3mpc_solve_batch_host")
        self.h_meta[3].fill_(-1)      # the host entry returns no task code (status carries the outcome)
        return self.h_out, self.h_meta

    def solve_host(self, p0, v0, goal) -> HostSolution:
        self.stage_host_inputs(p0, v0, goal)
        if self.rows_supported and self.B < 65536 and self.outputs == "all":
            return HostSolution.from_packed_rows(self.N, self.solve_rows().numpy().copy())
        if self.rows_supported and self.outputs == "solution":
            return HostSolution.from_solution_rows(self.N, self.solve_rows().numpy().copy(), self.params)
        h_out, h_meta = self.solve_staged()
        return HostSolution.from_blocks(self.N, h_out.numpy()[:, : self.B], h_meta.numpy()[:, : self.B])


def extract_batch(thrust_vectors, config: Optional[SE3MPCConfig] = None, *, mass: float = 1.5,
                  gravity: float = 9.81, dt: Optional[float] = None, untilted: bool = False):
    """`_extract_solution_from_result` (se3_mpc_planner.py:582-654) for B thrust sequences on the
    GPU: (B, N, 3) thrust vectors -> (accelerations, attitudes, body_rates, thrusts) host arrays
    of the reference's shapes.  The same device code as the solve kernel's epilogue."""
    torch = _torch()
    T = np.ascontiguousarray(thrust_vectors, np.float64)
    B, N, _ = T.shape
    cfg = config or SE3MPCConfig(prediction_horizon=N)
    params = make_params(cfg, mass=mass, gravity=gravity, dt=dt)
    if int(params.horizon) != N:
        raise ValueError("thrust_vectors must have config.prediction_horizon steps")
    ld = max(32, (B + 31) // 32 * 32)
    t_in = torch.zeros((3 * N, ld), dtype=torch.float64, device="cuda")
    t_in[:, :B] = torch.as_tensor(T.reshape(B, 3 * N)).cuda().t()
    out = torch.zeros((10 * N, ld), dtype=torch.float64, device="cuda")
    es = 8 * ld
    rc = _cabi.lib().dart_se3mpc_extract_batch(
        C.byref(params), B, ld, t_in.data_ptr(), out.data_ptr(), out.data_ptr() + 3 * N * es,
        out.data_ptr() + 6 * N * es, out.data_ptr() + 9 * N * es, 1 if untilted else 0,
        torch.cuda.current_stream().cuda_stream)
    _cabi.check(rc, "dart_se3mpc_extract_batch")
    h = out[:, :B].t().contiguous().cpu().numpy()
    return (h[:, : 3 * N].reshape(B, N, 3), h[:, 3 * N: 6 * N].reshape(B, N, 3),
            h[:, 6 * N: 9 * N].reshape(B, N, 3), h[:, 9 * N:])


class steps_in_flight:
    """Context manager for a caller that keeps several batched solves in flight on different CUDA
    streams (a planning server working through a stream of steps): tells the library how many
    problems that is in total, so the build is chosen for the machine's real load instead of one
    launch's B (`dart_se3mpc_set_inflight_hint`).  Four 4 096-problem steps in flight run at
    14.4 us per step on a B200; one at a time takes 24.7 us.

    >>> with dp.planner.steps_in_flight(4 * B):
    ...     for k, ws in enumerate(workspaces):           # resident inputs, one workspace per step
    ...         ws.solve_device(streams[k % 4])
    """

    def __init__(self, problems: int):
        self.problems = int(problems)

    def __enter__(self):
        _cabi.check(_cabi.lib().dart_se3mpc_set_inflight_hint(self.problems), "dart_se3mpc_set_inflight_hint")
        return self

    def __exit__(self, *exc):
        _cabi.lib().dart_se3mpc_set_inflight_hint(0)
        return False


def plan_batch(positions, velocities, goals, config: Optional[SE3MPCConfig] = None, *,
               mass: float = 1.5, gravity: float = 9.81, dt: Optional[float] = None,
               has_goal=None, x_warm=None, warm_mask=None, gradient_mode: int = 0,
               device=None, outputs: str = "all", to_host: bool = False, grid=None,
               safety_margin: float = 1.0, collision_threshold: float = 0.6,
               obstacle_penalty: bool = False, dynamics_consistent: bool = False, penalty_grid=None,
               spheres=None, sphere_margin: Optional[float] = None, reference=None):
    """Solve B independent SE(3)-MPC problems in one call.

    positions, velocities, goals : (B, 3) array-likes (NumPy or torch, host or device)
    config : SE3MPCConfig; ``config.dt`` is used as-is unless ``dt`` is given (the batched API
             exposes dt explicitly; only the drop-in class applies the reference's 1/400 s
             override)
    x_warm : (B, 9N) previous solutions for warm starts (se3_mpc_planner.py:294-327)
    grid   : DenseOccupancyGrid; adds the fused post-hoc `is_trajectory_safe` check of every
             solved trajectory (result.first_hit / result.safe)
    obstacle_penalty : with a grid, also add the occupancy-grid obstacle penalty to the objective
             and gradient inside the solve (gradient_mode 2; extension -- the reference solve has
             no obstacle term; weight = config.obstacle_weight, free level = the grid's prior)
    dynamics_consistent : optimise the thrusts only; positions and velocities are the rollout of
             the plant model from (p0, v0) (gradient_mode 3, with ``obstacle_penalty`` mode 4;
             extension).  The P/V rows of the result are that rollout; ``pos_bound`` and
             ``max_velocity`` are not enforced in this mode.
    penalty_grid : DenseOccupancyGrid the obstacle penalty reads instead of ``grid`` (typically
             ``grid.clearance_field(d_safe)``; free level = its prior).  ``grid``, if given, is then
             only the safety check's, run as a second launch on the solved positions.
    spheres : (centers (S, 3), radii (S,)), NumPy or torch: the sphere obstacle penalty in the solve
             (gradient_mode 5, with ``dynamics_consistent`` mode 6; extension -- the quadratic
             penalty of the reference's constraint |P_k - c|^2 >= (r + safety_margin)^2, weight
             ``config.obstacle_weight``; definition in include/dart_se3mpc.h, dart_spheres).  One list
             for the whole batch, uploaded once per call.  ``grid`` then only adds the safety check.
    sphere_margin : added to every radius; default ``config.safety_margin``.
    reference : (P (B, N, 3), V (B, N, 3) or None = zero velocities), NumPy or torch, host or device:
             track a per-timestep reference instead of flying to a goal (gradient_mode 7, with
             ``spheres`` mode 8; extension; definition in include/dart_se3mpc.h, dart_track_ref).
             Needs ``dynamics_consistent=True``; ``goals`` may then be None and is not read.
    Returns a BatchSolution (device) or HostSolution (``to_host=True``).
    """
    cfg = config or SE3MPCConfig()
    if reference is not None:
        if not dynamics_consistent:
            raise ValueError("reference= tracks with the dynamics-consistent solve: pass dynamics_consistent=True")
        if obstacle_penalty or penalty_grid is not None:
            raise ValueError("reference= does not combine with the grid penalty (obstacle_penalty)")
    elif goals is None:
        raise ValueError("goals may be None only with reference=")
    if dynamics_consistent:
        if gradient_mode != 0:
            raise ValueError("dynamics_consistent selects its own gradient mode")
        gradient_mode = 3
    if spheres is not None:
        if obstacle_penalty or penalty_grid is not None:
            raise ValueError("spheres= is an obstacle penalty of its own: it does not combine with obstacle_penalty")
        if gradient_mode not in (0, 3):
            raise ValueError("spheres= needs the reference gradient mode (or dynamics_consistent=True)")
        gradient_mode = 5 if gradient_mode == 0 else 6
    if reference is not None:
        gradient_mode = 7 if gradient_mode == 3 else 8
    pen = penalty_grid if penalty_grid is not None else grid
    if obstacle_penalty:
        if pen is None or gradient_mode not in (0, 3):
            raise ValueError("obstacle_penalty needs grid= or penalty_grid= and the reference gradient mode")
        gradient_mode = 2 if gradient_mode == 0 else 4
    if penalty_grid is not None and not obstacle_penalty:
        raise ValueError("penalty_grid= is the obstacle penalty's grid: pass obstacle_penalty=True")
    params = make_params(cfg, mass=mass, gravity=gravity, dt=dt, gradient_mode=gradient_mode,
                         obstacle_free_level=pen.prob_prior if pen is not None else 0.5)
    B = int(np.shape(positions)[0])
    ws = BatchWorkspace(params, B, device=device, pinned=False, outputs=outputs)
    ws.set_inputs_device(positions, velocities, np.zeros((B, 3)) if goals is None else goals)
    ws.set_has_goal(has_goal)
    ws.set_warm(x_warm, warm_mask)
    if grid is not None or penalty_grid is not None:
        ws.set_map(grid, safety_margin, collision_threshold, penalty_grid=penalty_grid)
    if spheres is not None:
        ws.set_spheres(spheres, cfg.safety_margin if sphere_margin is None else sphere_margin)
    if reference is not None:
        P, V = reference
        if int(np.shape(P)[1]) != int(params.horizon):
            raise ValueError(f"reference= needs N = {int(params.horizon)} samples per problem, got {np.shape(P)[1]}")
        ws.set_reference(P, V)
    sol = ws.solve_device()
    return sol.numpy() if to_host else sol


# ======================================================================================
class SE3MPCPlanner:
    """Drop-in for the reference ``SE3MPCPlanner`` (se3_mpc_planner.py:82-757).

    Differences, all opt-in: ``store_last_solution=True`` keeps the previous solution so that
    the warm start of :294-327 actually runs (the reference never assigns ``last_solution``);
    ``control_frequency_hz`` selects the timing-alignment frequency whose inverse overrides
    ``config.dt`` (reference: always 400 Hz unless reconfigured, :99-122);
    ``avoid_obstacles=True`` makes the obstacle list (``add_obstacle``, ``update_plan``,
    ``refresh_obstacles_from_mapper``) enter the solve as the sphere penalty of gradient_mode 5 with
    ``config.safety_margin`` and ``config.obstacle_weight`` -- the reference builds that constraint
    and never passes it to ``minimize`` (:499-514), so by default the list changes nothing here either.
    """

    def __init__(self, config: Optional[SE3MPCConfig] = None, *, mass: float = 1.5,
                 control_frequency_hz: Optional[float] = None, respect_config_dt: bool = False,
                 store_last_solution: bool = False, device=None, avoid_obstacles: bool = False):
        if config is None:
            config = SE3MPCConfig()
        if control_frequency_hz is None:
            control_frequency_hz = float(os.environ.get("DART_CONTROL_FREQUENCY_HZ",
                                                        REFERENCE_CONTROL_FREQUENCY_HZ))
        aligned_dt = config.dt if respect_config_dt else 1.0 / control_frequency_hz
        d = config.as_dict()
        d["dt"] = aligned_dt
        self.se3_config = SE3MPCConfig(**d)
        self.config = AttrDict(d)
        self.mass = float(to_si(mass, "kg"))
        self.gravity = 9.81
        self.hover_thrust = self.mass * self.gravity
        self.goal_position: Optional[np.ndarray] = None
        self.obstacles: List[Tuple[np.ndarray, float]] = []
        self.last_solution: Optional[Dict[str, np.ndarray]] = None
        self.warm_start_enabled = True
        self.store_last_solution = store_last_solution
        self.planning_times: List[float] = []
        self.plan_count = 0
        self.convergence_history: List[bool] = []
        self.last_result: Dict[str, Any] = {}
        self.planning_stats = {"total_plans": 0, "successful_plans": 0, "planning_times": [],
                               "last_plan_time": 0.0}
        self.logger = logger
        self._params = make_params(self.se3_config, mass=self.mass, gravity=self.gravity)
        self.avoid_obstacles = bool(avoid_obstacles)
        self._params_spheres = make_params(self.se3_config, mass=self.mass, gravity=self.gravity, gradient_mode=5)
        self._device = device
        _cabi.lib()  # fail now, loudly, if the CUDA library is missing

    @classmethod
    def from_yaml(cls, defaults_path: Optional[str] = None, airframe: str = "default",
                  airframes_path: Optional[str] = None, **kw) -> "SE3MPCPlanner":
        """Planner configured from config/defaults.yaml (`planning:`) + config/airframes.yaml."""
        cfg, mass = load_planner_config(defaults_path, airframe, airframes_path)
        kw.setdefault("respect_config_dt", True)
        return cls(cfg, mass=mass, **kw)

    # ---- IPlanner / BasePlanner surface (common/interfaces.py:81-105, base_planner.py:16-112)
    def set_goal(self, goal_position) -> None:
        self.goal_position = np.array(to_si(goal_position, "m"), dtype=np.float64).reshape(3).copy()

    def add_obstacle(self, center, radius) -> None:
        self.obstacles.append((np.array(to_si(center, "m"), dtype=np.float64).reshape(3).copy(),
                               float(np.asarray(to_si(radius, "m")))))

    def clear_obstacles(self) -> None:
        self.obstacles.clear()

    def refresh_obstacles_from_mapper(self, mapper, center, size: float = 20.0, threshold: float = 0.6,
                                      max_spheres: int = 20, radius: float = 1.0) -> int:
        """The cloud node's mapper -> planner bridge (cloud/main_improved_threelayer.py:381-398):
        replace the obstacle list by spheres on the occupied sample points of the mapper's local
        grid.  Returns the number of spheres."""
        self.clear_obstacles()
        for c, r in mapper.occupied_spheres(center, size, threshold, max_spheres, radius):
            self.add_obstacle(c, r)
        return len(self.obstacles)

    def sense(self, current_state: DroneState, goal_position):
        goal = np.array(to_si(goal_position, "m"), dtype=np.float64).reshape(3)
        if self.goal_position is None or np.linalg.norm(self.goal_position - goal) > 0.5:
            self.set_goal(goal)  # 0.5 m hysteresis (:199)
        return current_state, self.goal_position, list(self.obstacles)

    def plan(self, current_state: DroneState) -> Dict[str, np.ndarray]:
        return self._solve_se3_mpc(current_state)

    def act(self, solution, current_state, start_time: float) -> Trajectory:
        return self._create_trajectory_from_solution(solution, start_time)

    def plan_trajectory(self, current_state: DroneState, goal_position) -> Trajectory:
        current_state, _, _ = self.sense(current_state, goal_position)
        solution = self.plan(current_state)
        return self.act(solution, current_state, time.time())

    def update_plan(self, current_state: DroneState, obstacles: Sequence[Dict[str, Any]]) -> Trajectory:
        self.clear_obstacles()
        for ob in obstacles:
            if "position" in ob and "radius" in ob:
                self.add_obstacle(np.array(ob["position"]), ob["radius"])
        if self.goal_position is not None:
            return self.plan_trajectory(current_state, self.goal_position)
        return self._generate_emergency_trajectory(current_state)

    def is_plan_valid(self, trajectory: Optional[Trajectory]) -> bool:
        if trajectory is None or len(trajectory.positions) == 0:
            return False
        P = np.asarray(trajectory.positions)
        if not np.all(np.isfinite(P)) or np.any(P[:, 2] < 0.1):
            return False
        if trajectory.velocities is not None and np.any(np.abs(np.asarray(trajectory.velocities)) > 20.0):
            return False
        return True

    def validate_goal(self, goal) -> bool:
        goal = None if goal is None else np.asarray(goal)
        return goal is not None and goal.shape == (3,) and not goal[2] < 0.5

    def validate_state(self, state: Optional[DroneState]) -> bool:
        if state is None or not np.all(np.isfinite(state.position)):
            return False
        return not np.any(np.abs(state.velocity) > 20.0)

    def get_planning_stats(self) -> Dict[str, Any]:
        if not self.planning_times:
            return {}
        return {"mean_planning_time_ms": float(np.mean(self.planning_times)),
                "max_planning_time_ms": float(np.max(self.planning_times)),
                "success_rate": float(np.mean(self.convergence_history)) if self.convergence_history else 0.0,
                "total_plans": self.plan_count}

    def reset_performance_tracking(self) -> None:
        self.planning_times.clear()
        self.convergence_history.clear()
        self.plan_count = 0

    def get_config(self) -> SE3MPCConfig:
        return self.se3_config

    # ---- the solve (:230-280) ---------------------------------------------------------------
    def _solve_se3_mpc(self, current_state: DroneState) -> Dict[str, np.ndarray]:
        N = self.se3_config.prediction_horizon
        L = _cabi.lib()
        t0 = time.perf_counter()
        p0 = np.ascontiguousarray(current_state.position, np.float64)
        v0 = np.ascontiguousarray(current_state.velocity, np.float64)
        has_goal = self.goal_position is not None
        goal = np.ascontiguousarray(self.goal_position if has_goal else np.zeros(3), np.float64)
        hg = np.array([1 if has_goal else 0], np.uint8)
        xw = None
        if self.warm_start_enabled and self.last_solution is not None:
            prev = self.last_solution
            if len(prev["positions"]) == N:
                xw = np.ascontiguousarray(np.concatenate([
                    np.asarray(prev["positions"]).ravel(), np.asarray(prev["velocities"]).ravel(),
                    np.asarray(prev["thrust_vectors"]).ravel()]), np.float64)
            else:
                raise ValueError("warm start needs a previous solution of the same horizon")
        out = np.empty(out_rows(N), np.float64)
        meta = np.zeros(3, np.int32)
        vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        o = out.ctypes.data
        args = (1, vp(p0), vp(v0), vp(goal), vp(hg), None if xw is None else vp(xw),
                o, o + 8 * 9 * N, meta.ctypes.data, meta.ctypes.data + 4, meta.ctypes.data + 8,
                o + 8 * (9 * N + 1), o + 8 * (12 * N + 1), o + 8 * (15 * N + 1), o + 8 * (18 * N + 1))
        if self.avoid_obstacles and self.obstacles:
            rows = np.ascontiguousarray([[*c, r] for c, r in self.obstacles], np.float64)
            sph = _cabi.Spheres(len(rows), 0, rows.ctypes.data, float(self.se3_config.safety_margin))
            rc = L.dart_se3mpc_solve_batch_host_spheres(C.byref(self._params_spheres), *args, C.byref(sph))
            _cabi.check(rc, "dart_se3mpc_solve_batch_host_spheres")
        else:
            rc = L.dart_se3mpc_solve_batch_host(C.byref(self._params), *args)
            _cabi.check(rc, "dart_se3mpc_solve_batch_host")
        converged = bool(meta[2] == 0)
        self.convergence_history.append(converged)
        if not converged:
            self.logger.warning("SE(3) MPC optimization did not converge (status %d)", int(meta[2]))
        solution = {
            "positions": out[0:3 * N].reshape(N, 3),
            "velocities": out[3 * N:6 * N].reshape(N, 3),
            "thrust_vectors": out[6 * N:9 * N].reshape(N, 3),
            "accelerations": out[9 * N + 1:12 * N + 1].reshape(N, 3),
            "attitudes": out[12 * N + 1:15 * N + 1].reshape(N, 3),
            "body_rates": out[15 * N + 1:18 * N + 1].reshape(N, 3),
            "thrusts": out[18 * N + 1:19 * N + 1],
        }
        self.last_result = {"fun": float(out[9 * N]), "nit": int(meta[0]), "nfev": int(meta[1]),
                            "status": int(meta[2]), "success": converged, "x": out[:9 * N]}
        if self.store_last_solution:
            self.last_solution = {k: solution[k].copy() for k in ("positions", "velocities", "thrust_vectors")}
        dt_ms = (time.perf_counter() - t0) * 1e3
        self.planning_times.append(dt_ms)
        self.plan_count += 1
        return solution

    def _create_trajectory_from_solution(self, solution, start_time: float) -> Trajectory:
        N = len(solution["positions"])
        timestamps = start_time + np.arange(N) * self.se3_config.dt
        return Trajectory(timestamps=timestamps, positions=solution["positions"],
                          velocities=solution["velocities"], accelerations=solution["accelerations"],
                          attitudes=solution["attitudes"], body_rates=solution["body_rates"],
                          thrusts=solution["thrusts"], yaws=solution["attitudes"][:, 2],
                          yaw_rates=solution["body_rates"][:, 2])

    def _generate_emergency_trajectory(self, current_state: DroneState) -> Trajectory:
        N, dt = self.se3_config.prediction_horizon, self.se3_config.dt
        return Trajectory(timestamps=current_state.timestamp + np.arange(N) * dt,
                          positions=np.tile(current_state.position, (N, 1)),
                          velocities=np.zeros((N, 3)), accelerations=np.zeros((N, 3)))

    # ---- batched entry on the same configuration ---------------------------------------------
    def plan_batch(self, positions, velocities, goals, **kw):
        """Batched solve with this planner's configuration, mass and (aligned) dt."""
        kw.setdefault("mass", self.mass)
        kw.setdefault("gravity", self.gravity)
        kw.setdefault("device", self._device)
        return plan_batch(positions, velocities, goals, self.se3_config, **kw)


class PlannerFactory:
    """Same registry shape as planning/base_planner.py:114-136."""

    _planners: Dict[str, type] = {}

    @classmethod
    def register(cls, name: str, planner_class: type) -> None:
        cls._planners[name] = planner_class

    @classmethod
    def create(cls, name: str, config=None):
        if name not in cls._planners:
            raise ValueError(f"Unknown planner type: {name}")
        if isinstance(config, dict):
            config = SE3MPCConfig(**config)
        return cls._planners[name](config)

    @classmethod
    def list_planners(cls) -> List[str]:
        return list(cls._planners)


PlannerFactory.register("se3_mpc", SE3MPCPlanner)  # se3_mpc_planner.py:760-762
