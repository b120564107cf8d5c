"""Closed-loop receding-horizon simulation on resident device state (BASELINE configs[4]).

Every drone replans at a fixed rate: solve from the current (p, v) with the warm start of
se3_mpc_planner.py:294-327 (the reference builds it but never stores `last_solution`; here the
previous solution is kept, SURVEY.md 8(d).5), then the state advances with the planner's own
model (:430-431, :445-459) driven by the first control of the new solution.  One kernel launch
per replanning step for the whole population (`dart_se3mpc_closed_loop_step`): state, goals and
solutions never leave HBM; only what the caller asks for is copied out.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _cabi


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("dart_planner_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch


class ClosedLoopSim:
    """B drones, fixed goals, replanning every `plant_dt` seconds.

    >>> sim = ClosedLoopSim(params, B, plant_dt=0.1)
    >>> sim.reset(p0, v0, goals)
    >>> sim.run(100)                  # 100 launches, state stays on the device
    >>> sim.positions(), sim.velocities(), sim.nfev_total

    Dynamics-consistent params (gradient_mode 3) are accepted: the plan's positions and velocities
    are then the rollout of the same plant model, so with ``plant_dt == params.dt`` the state after
    a step is the plan's P_1 / V_1.  Warm starts use the 9-slot kernel (the lateral thrust moves).

    Against a map (``dart_se3mpc_closed_loop_step_map``):
      penalty_grid  : DenseOccupancyGrid the obstacle penalty of gradient_mode 2 / 4 reads (those
                      modes need it; typically ``grid.clearance_field(d_safe)``; params'
                      ``obstacle_free_level`` should be its prior, 0.5)
      collision_map : DenseOccupancyGrid the flown path of every step is checked against: the
                      straight segment from the state before to the state after the step, sampled
                      at steps of at most half a voxel (at most 64 samples), each sample with
                      is_trajectory_safe's stencil (``safety_margin``, ``collision_threshold``).
                      ``first_collision()`` is the first step index at which a drone's path
                      collided, -1 = never.
      spheres       : (centers (S, 3), radii (S,)): the sphere obstacle penalty of gradient_mode 5
                      (mode 0 + spheres) or 6 (mode 3 + spheres), which need it, every radius
                      inflated by ``sphere_margin`` (``dart_se3mpc_closed_loop_step_spheres``; a
                      ``collision_map`` still judges collisions, typically the same spheres
                      rasterised by ``add_obstacles``).  Mode 5 keeps the lateral thrust at exactly
                      zero, so its warm starts use the 7-slot kernel as in mode 0.

    Tracking a path (``dart_se3mpc_closed_loop_step_track``):
      reference_path : (P (B, T, 3), V (B, T, 3) or None = zero velocities), NumPy or torch: the
                      per-timestep reference of gradient_mode 7 (mode 3 tracking it) or 8 (mode 6
                      tracking it, with ``spheres``), which need it.  Uploaded once; step s tracks
                      samples s, s+1, .., s+N-1, the last sample held past the end of the path, so
                      the window slides one sample per replan (``plant_dt`` must equal ``params.dt``).
                      ``mission.reference_path`` samples one from waypoints.  Goals are not read.
    """

    def __init__(self, params: _cabi.Params, B: int, plant_dt: Optional[float] = None, device=None, *,
                 penalty_grid=None, collision_map=None, safety_margin: float = 0.0,
                 collision_threshold: float = 0.6, spheres=None, sphere_margin: float = 0.0,
                 reference_path=None):
        gm = int(params.gradient_mode)
        if gm in (2, 4) and penalty_grid is None:
            raise ValueError("ClosedLoopSim: gradient_mode 2 / 4 need penalty_grid=")
        if (gm in (5, 6, 8)) != (spheres is not None):
            raise ValueError("ClosedLoopSim: spheres= goes with gradient_mode 5 / 6 / 8, and they need it")
        if (gm in (7, 8)) != (reference_path is not None):
            raise ValueError("ClosedLoopSim: reference_path= goes with gradient_mode 7 / 8, and they need it")
        if reference_path is not None and float(params.dt if plant_dt is None else plant_dt) != float(params.dt):
            raise ValueError("ClosedLoopSim: reference_path= slides one sample per step: plant_dt must equal dt")
        torch = _torch()
        self.penalty_grid, self.collision_map = penalty_grid, collision_map
        self.safety_margin, self.collision_threshold = float(safety_margin), float(collision_threshold)
        self.params = params
        self.N = int(params.horizon)
        self.B = int(B)
        self.ld = max(32, (self.B + 31) // 32 * 32)
        self.plant_dt = float(params.dt if plant_dt is None else plant_dt)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.spheres = self._spheres_dev = None
        if spheres is not None:
            from .planner import sphere_rows
            rows = sphere_rows(spheres)
            self._spheres_dev = torch.as_tensor(rows).to(self.device) if len(rows) else None
            self.spheres = _cabi.Spheres(len(rows), 0, None if self._spheres_dev is None
                                         else self._spheres_dev.data_ptr(), float(sphere_margin))
        self._ref_rows = None
        if reference_path is not None:
            from .planner import reference_rows
            P, V = reference_path
            self._ref_rows = reference_rows(P, V, self.B, self.ld, self.device)
        f8 = dict(dtype=torch.float64, device=self.device)
        self.state = torch.zeros((9, self.ld), **f8)            # rows p xyz | v xyz | goal xyz
        self.x = torch.zeros((9 * self.N, self.ld), **f8)       # current solution, reference order
        self.cost = torch.zeros(self.ld, **f8)
        self.meta = torch.zeros((3, self.ld), dtype=torch.int32, device=self.device)  # nit, nfev, status
        self.nfev_total = torch.zeros(self.ld, dtype=torch.int64, device=self.device)
        self._first_collision = torch.full((self.ld,), -1, dtype=torch.int32, device=self.device)
        self.steps_done = 0
        # the solutions held in self.x come from cold starts of this solver, so their lateral
        # thrust is exactly zero and stays zero: warm starts may use the 7-slot kernel (warm=2;
        # the kernel verifies).  Anyone writing self.x by hand must clear this flag.
        self.lateral_thrust_is_zero = self._untilted_mode()
        self._lib = _cabi.lib()

    def _untilted_mode(self) -> bool:
        """Modes whose cold-started lateral thrust stays exactly zero (all but the dynamics-consistent
        modes 3, 4, 6, 7 and 8)."""
        return int(self.params.gradient_mode) in (0, 1, 2, 5)

    def reset(self, p0, v0, goals=None):
        """Initial states; ``goals`` (B, 3), which the tracking modes 7 / 8 do not read (None: zeros)."""
        torch = _torch()
        if goals is None:
            if self._ref_rows is None:
                raise ValueError("ClosedLoopSim.reset: goals are needed without reference_path=")
            goals = np.zeros((self.B, 3))
        for i, a in enumerate((p0, v0, goals)):
            t = torch.as_tensor(np.asarray(a, np.float64) if not torch.is_tensor(a) else a,
                                dtype=torch.float64).to(self.device)
            self.state[3 * i: 3 * i + 3, : self.B] = t.reshape(self.B, 3).t()
        self.x.zero_()
        self.nfev_total.zero_()
        self._first_collision.fill_(-1)
        self.steps_done = 0
        self.lateral_thrust_is_zero = self._untilted_mode()

    def _launch(self, lo: int, hi: int, stream, track_counters: bool):
        """One replanning step of drones [lo, hi) (one launch): solve, store, advance the plant."""
        torch = _torch()
        es = 8 * self.ld
        base = self.state.data_ptr() + 8 * lo
        meta = self.meta.data_ptr() + 4 * lo
        args = (C.byref(self.params), hi - lo, self.ld, base, base + 3 * es, base + 6 * es, None,
                self.x.data_ptr() + 8 * lo,
                0 if self.steps_done == 0 else (2 if self.lateral_thrust_is_zero else 1), self.cost.data_ptr() + 8 * lo,
                meta, meta + 4 * self.ld, meta + 8 * self.ld, self.plant_dt)
        with torch.cuda.device(self.device):
            cg = self.collision_map._grid() if self.collision_map is not None else None
            record = (C.byref(cg) if cg is not None else None, self.safety_margin, self.collision_threshold,
                      self.steps_done, self._first_collision.data_ptr() + 4 * lo if cg is not None else None,
                      stream.cuda_stream)
            if self._ref_rows is not None:
                name = "dart_se3mpc_closed_loop_step_track"
                ref = _cabi.TrackRef(self._ref_rows.shape[0] // 6, self.steps_done, self._ref_rows.data_ptr() + 8 * lo)
                rc = self._lib.dart_se3mpc_closed_loop_step_track(
                    *args[:5], *args[6:], C.byref(ref), None if self.spheres is None else C.byref(self.spheres),
                    *record)
            elif self.spheres is not None:
                name = "dart_se3mpc_closed_loop_step_spheres"
                rc = self._lib.dart_se3mpc_closed_loop_step_spheres(*args, C.byref(self.spheres), *record)
            elif self.penalty_grid is None and self.collision_map is None:
                name = "dart_se3mpc_closed_loop_step"
                rc = self._lib.dart_se3mpc_closed_loop_step(*args, stream.cuda_stream)
            else:
                name = "dart_se3mpc_closed_loop_step_map"
                pg = self.penalty_grid._grid() if self.penalty_grid is not None else None
                rc = self._lib.dart_se3mpc_closed_loop_step_map(
                    *args, C.byref(pg) if pg is not None else None, *record)
        _cabi.check(rc, name)
        if track_counters:
            with torch.cuda.stream(stream):
                self.nfev_total[lo:hi] += self.meta[1, lo:hi]

    def step(self, stream=None, track_counters: bool = True):
        """One replanning step of the whole population (one launch)."""
        torch = _torch()
        self._launch(0, self.B, stream or torch.cuda.current_stream(self.device), track_counters)
        self.steps_done += 1

    def default_parts(self) -> int:
        """Sub-populations `run` keeps in flight (measured, tools/closed_loop_parts.py, 100 replans on
        one B200, ms for 1 / 2 / 3 / 4 parts): 65 536 drones 22.0 / 21.6 / 21.6 / 21.7; 32 768: 11.5 /
        10.8 / 10.8 / 11.1; 16 384: 6.8 / 5.6 / 5.5 / 5.6; 8 192 (one GPU's share of 65 536 on eight):
        4.6 / 3.5 / 3.3 / 3.6 -- the fewer waves of blocks a step has, the more its idle tail costs."""
        return 2 if self.B >= 49152 else (3 if self.B >= 6144 else 1)

    def run(self, steps: int, stream=None, track_counters: bool = True, record: bool = False,
            parts: Optional[int] = None):
        """`steps` replans.  record=True returns the (steps, B, 3) position history (host).

        A drone's step k+1 depends on ITS step k only, so the population is replanned as `parts`
        independent sub-populations (contiguous index ranges, a CUDA stream each): while the last,
        partly filled wave of one sub-population's step drains, the next step of another one
        already fills the free SMs -- with one launch per step for everybody, every step ends
        with that idle tail (65 536 drones: 9.2 waves of blocks per step; 8 192 per GPU on eight
        GPUs: 1.15).  Same launches, same results per drone; only their order on the machine
        changes.  The library is told how many problems are in flight so that the sub-population
        launches are served by the throughput build like the whole population would be."""
        torch = _torch()
        stream = stream or torch.cuda.current_stream(self.device)
        parts = self.default_parts() if parts is None else max(1, int(parts))
        if record or parts == 1 or steps <= 0:
            hist = []
            for _ in range(steps):
                self.step(stream, track_counters)
                if record:
                    hist.append(self.positions().cpu().numpy())
            return np.stack(hist) if record else None
        # contiguous ranges, multiples of 64 drones (whole 512-byte row segments)
        per = (self.B // parts + 63) // 64 * 64
        ranges = [(a, min(a + per, self.B)) for a in range(0, self.B, per)]
        if getattr(self, "_side", None) is None or len(self._side) < len(ranges) - 1:
            self._side = [torch.cuda.Stream(self.device) for _ in range(len(ranges) - 1)]
        streams = [stream] + self._side[: len(ranges) - 1]
        start = torch.cuda.Event()
        start.record(stream)
        for st in streams[1:]:
            st.wait_event(start)
        self._lib.dart_se3mpc_set_inflight_hint(self.B)
        try:
            for _ in range(steps):
                for (lo, hi), st in zip(ranges, streams):
                    self._launch(lo, hi, st, track_counters)
                self.steps_done += 1
        finally:
            self._lib.dart_se3mpc_set_inflight_hint(0)
        for st in streams[1:]:
            done = torch.cuda.Event()
            done.record(st)
            stream.wait_event(done)
        return None

    def first_collision(self):
        """(B,) int32: the step index (``steps_done`` when it ran) of each drone's first collision
        with ``collision_map``, -1 = never (always -1 without a collision map)."""
        return self._first_collision[: self.B]

    def positions(self):
        return self.state[0:3, : self.B].t()

    def velocities(self):
        return self.state[3:6, : self.B].t()

    def goals(self):
        return self.state[6:9, : self.B].t()

    def solution(self):
        """(B, 9N) current solutions in the reference's packed order."""
        return self.x[:, : self.B].t()
