"""Dense device occupancy grid with the query surface of the reference's
``ExplicitGeometricMapper`` (perception/explicit_geometric_mapper.py), batched.

The reference keeps a sparse dict keyed by ``floor(p / resolution)`` with prior 0.5 for
unknown voxels (:154-169).  Here the map is a dense fp32 grid [nz][ny][nx] resident in HBM
(256^3 = 64 MiB, L2-resident on B200); keys outside the grid read the prior, as a dict miss.
"""
from __future__ import annotations

import ctypes as C
import time
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Tuple

import numpy as np

from . import _cabi


@dataclass
class SensorObservation:
    """One range measurement (explicit_geometric_mapper.py:29-37)."""
    position: np.ndarray
    direction: np.ndarray
    hit_distance: Optional[float]
    max_range: float
    timestamp: float = 0.0


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("dart_planner_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch


class DenseOccupancyGrid:
    def __init__(self, shape: Tuple[int, int, int] = (256, 256, 256),
                 origin_voxel: Tuple[int, int, int] = (-128, -128, -128),
                 resolution: float = 0.2, prior: float = 0.5, device=None, max_range: float = 50.0,
                 dtype: str = "float32"):
        """dtype "float32" (default: half the bytes; probabilities carry 1e-7 of rounding, e.g. a
        single miss reads 0.60000002 instead of the reference's 0.6) or "float64" (the reference's
        own precision: its voxels hold Python floats)."""
        torch = _torch()
        if dtype not in ("float32", "float64"):
            raise ValueError("dtype must be 'float32' or 'float64'")
        self.dtype = dtype
        self.nx, self.ny, self.nz = (int(s) for s in shape)
        self.origin_voxel = tuple(int(o) for o in origin_voxel)
        self.resolution = float(resolution)
        self.prob_prior = float(prior)
        self.prob_hit, self.prob_miss = 0.7, 0.4        # explicit_geometric_mapper.py:80-81
        self.max_range = float(max_range)               # :66
        self.total_observations = 0
        self._counts = None                              # update_map scratch (uint64 per cell)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.occ = torch.full((self.nz, self.ny, self.nx), prior, device=self.device,
                              dtype=torch.float64 if dtype == "float64" else torch.float32)

    # -- plumbing ------------------------------------------------------------------------
    def _grid(self) -> _cabi.Grid:
        return _cabi.Grid(self.nx, self.ny, self.nz, *self.origin_voxel, self.resolution,
                          self.prob_prior, self.occ.data_ptr(), 8 if self.dtype == "float64" else 4, 0)

    def _stream(self, stream):
        torch = _torch()
        return (stream or torch.cuda.current_stream(self.device)).cuda_stream

    def _soa(self, a, rows):
        """(B, rows) array-like -> contiguous (rows, B) float64 device tensor."""
        torch = _torch()
        t = torch.as_tensor(np.asarray(a, np.float64) if not torch.is_tensor(a) else a,
                            dtype=torch.float64).to(self.device)
        return t.reshape(-1, rows).t().contiguous()

    # -- reference surface -----------------------------------------------------------------
    def world_to_voxel(self, position) -> Tuple[int, int, int]:
        return tuple(int(v) for v in np.floor(np.asarray(position, float) / self.resolution).astype(int))

    def add_obstacle(self, center, radius: float, value: float = 0.9) -> None:
        self.add_obstacles(np.asarray(center, float).reshape(1, 3), [radius], value)

    def add_obstacles(self, centers, radii, value: float = 0.9, stream=None) -> None:
        """Rasterise spheres exactly like add_obstacle (:399-423)."""
        torch = _torch()
        c = self._soa(centers, 3)
        r = torch.as_tensor(np.asarray(radii, np.float64), dtype=torch.float64).to(self.device).contiguous()
        g = self._grid()
        rc = _cabi.lib().dart_map_add_spheres(C.byref(g), self.occ.data_ptr(), int(r.numel()),
                                              c.data_ptr(), r.data_ptr(), float(value), self._stream(stream))
        _cabi.check(rc, "dart_map_add_spheres")

    def query_occupancy_batch(self, positions, stream=None):
        """positions (B,3) -> (B,) float64 device tensor (query_occupancy_batch :171-182)."""
        torch = _torch()
        pos = self._soa(positions, 3)
        B = pos.shape[1]
        out = torch.empty(B, dtype=torch.float64, device=self.device)
        g = self._grid()
        rc = _cabi.lib().dart_map_query_batch(C.byref(g), B, B, pos.data_ptr(), out.data_ptr(),
                                              self._stream(stream))
        _cabi.check(rc, "dart_map_query_batch")
        return out

    def query_occupancy(self, position) -> float:
        return float(self.query_occupancy_batch(np.asarray(position, float).reshape(1, 3))[0])

    def is_collision(self, position, threshold: float = 0.6) -> bool:
        return self.query_occupancy(position) > threshold

    def trajectories_safe_soa(self, positions_soa, B: int, npos: int, safety_margin: float = 1.0,
                              threshold: float = 0.6, out=None, stream=None):
        """positions_soa: (3*npos, ld) device tensor with rows 3k+c (e.g. the first 3N rows of a
        BatchSolution.out) -> (ld,) int32 first-collision index, -1 = safe."""
        torch = _torch()
        ld = positions_soa.shape[1]
        assert positions_soa.is_cuda and positions_soa.dtype == torch.float64 and positions_soa.is_contiguous()
        assert positions_soa.shape[0] >= 3 * npos
        if out is None:
            out = torch.empty(ld, dtype=torch.int32, device=self.device)
        g = self._grid()
        rc = _cabi.lib().dart_map_traj_safe_batch(C.byref(g), B, ld, npos, positions_soa.data_ptr(),
                                                  float(safety_margin), float(threshold),
                                                  out.data_ptr(), self._stream(stream))
        _cabi.check(rc, "dart_map_traj_safe_batch")
        return out

    def are_trajectories_safe(self, positions, safety_margin: float = 1.0, threshold: float = 0.6):
        """positions (B, npos, 3) -> (B,) int32 first-collision index, -1 = safe."""
        torch = _torch()
        t = torch.as_tensor(np.asarray(positions, np.float64) if not torch.is_tensor(positions) else positions,
                            dtype=torch.float64).to(self.device)
        B, npos, _ = t.shape
        soa = t.reshape(B, 3 * npos).t().contiguous()
        return self.trajectories_safe_soa(soa, B, npos, safety_margin, threshold)[:B]

    def is_trajectory_safe(self, positions, safety_margin: float = 1.0, threshold: float = 0.6):
        """Reference signature (:195-219): returns (is_safe, first_collision_index)."""
        idx = int(self.are_trajectories_safe(np.asarray(positions, float)[None], safety_margin, threshold)[0])
        return idx < 0, idx

    def update_map(self, positions, directions=None, hit_distances=None, max_ranges=50.0, stream=None,
                   sync: bool = True):
        """Batched `update_map` (:100-152) for one scan.  Either the reference's argument -- a list
        of SensorObservation (position / direction / hit_distance / max_range; hit_distance None
        = no return) -- or the same as arrays / device tensors ((B,3), (B,3), (B,), scalar or (B,);
        NaN = no return).  Two launches: ray walk with per-voxel visit counters, then the Bayes
        rule applied per voxel.  Returns the reference's counters dict; with ``sync=False`` nothing
        is read back (no host synchronisation: the counters stay device tensors, `total_voxels`
        is left out), which is what a scan-rate caller with device-resident point clouds uses."""
        torch = _torch()
        if directions is None:      # the reference's signature: update_map(observations)
            obs = list(positions)
            if not obs:
                return {"updated_voxels": 0, "observations_processed": 0,
                        "total_voxels": int((self.occ != self.prob_prior).sum().item())}
            positions = np.array([np.asarray(o.position, np.float64) for o in obs])
            directions = np.array([np.asarray(o.direction, np.float64) for o in obs])
            hit_distances = np.array([np.nan if o.hit_distance is None else float(o.hit_distance) for o in obs])
            max_ranges = np.array([float(o.max_range) for o in obs])
        start = self._soa(positions, 3)
        d = self._soa(directions, 3)
        B = start.shape[1]
        if torch.is_tensor(hit_distances):
            hit_t = hit_distances.to(self.device, torch.float64).reshape(-1)
        else:
            hd = np.asarray(hit_distances)
            if hd.dtype == object:      # the reference's Optional[float] per observation: None = no return
                hd = np.array([np.nan if h is None else float(h) for h in hd.reshape(-1)])
            hit_t = torch.as_tensor(np.ascontiguousarray(hd, np.float64).reshape(-1)).to(self.device)
        if torch.is_tensor(max_ranges):
            mr = max_ranges.to(self.device, torch.float64).reshape(-1).expand(B).contiguous()
        else:
            mr = torch.as_tensor(np.broadcast_to(np.asarray(max_ranges, np.float64), (B,)).copy()).to(self.device)
        updated = self.update_map_soa(start, d, hit_t, mr, stream)
        self.total_observations += B
        self.last_update_time = time.time()
        if not sync:
            return {"updated_voxels": updated, "observations_processed": B}
        return {"updated_voxels": int(updated.item()), "observations_processed": B,
                "total_voxels": int((self.occ != self.prob_prior).sum().item())}

    def update_map_soa(self, start_soa, dir_soa, hit, max_ranges, stream=None):
        """Lowest level: (3, B) float64 device tensors (rows x/y/z), (B,) hit distances (NaN = no
        return) and (B,) per-observation max ranges, all resident.  Two launches, no allocation
        after the first call, no synchronisation; returns the device counter of voxel visits."""
        torch = _torch()
        B = start_soa.shape[1]
        for t in (start_soa, dir_soa, hit, max_ranges):
            assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()
        if self._counts is None:
            self._counts = torch.zeros(self.nx * self.ny * self.nz, dtype=torch.int64, device=self.device)
            self._updated = torch.zeros(1, dtype=torch.int64, device=self.device)
        s = stream or torch.cuda.current_stream(self.device)
        with torch.cuda.stream(s):
            self._updated.zero_()
        g = self._grid()
        rc = _cabi.lib().dart_map_update_batch(
            C.byref(g), self.occ.data_ptr(), self._counts.data_ptr(), B, B, start_soa.data_ptr(), dir_soa.data_ptr(),
            hit.data_ptr(), max_ranges.data_ptr(), self.max_range, self.prob_hit, self.prob_miss,
            self._updated.data_ptr(), s.cuda_stream)
        _cabi.check(rc, "dart_map_update_batch")
        return self._updated

    def simulate_lidar_scan(self, drone_state, num_rays: int = 360) -> List[SensorObservation]:
        """The reference's test scan (:365-397): `num_rays` horizontal rays from the drone, each
        with a 10 % chance of a return at U(2, 20) m (NumPy's global generator, as there)."""
        observations = []
        for i in range(num_rays):
            angle = 2 * np.pi * i / num_rays
            direction = np.array([np.cos(angle), np.sin(angle), 0.0])
            hit_distance = np.random.uniform(2.0, 20.0) if np.random.random() < 0.1 else None
            observations.append(SensorObservation(position=np.asarray(drone_state.position, np.float64),
                                                  direction=direction, hit_distance=hit_distance,
                                                  max_range=self.max_range, timestamp=time.time()))
        return observations

    def get_local_occupancy_grid(self, center, size: float = 20.0) -> Tuple[np.ndarray, np.ndarray]:
        """:221-248: a cube of `int(size / resolution)`^3 sample points around `center`
        (`linspace` per axis, NumPy's meshgrid order) and their occupancies ->
        (positions (n, n, n, 3), occupancy (n, n, n)) host arrays; the occupancies are one batched
        query on the device."""
        center = np.asarray(getattr(center, "magnitude", center), np.float64).reshape(3)
        half = size / 2
        lo, hi = center - half, center + half
        n = int(size / self.resolution)
        x, y, z = (np.linspace(lo[c], hi[c], n) for c in range(3))
        pts = np.array(np.meshgrid(x, y, z)).T.reshape(-1, 3)
        occ = self.query_occupancy_batch(pts).cpu().numpy()
        return pts.reshape(n, n, n, 3), occ.reshape(n, n, n)

    def occupied_spheres(self, center, size: float = 20.0, threshold: float = 0.6, max_spheres: int = 20,
                         radius: float = 1.0) -> List[Tuple[np.ndarray, float]]:
        """The mapper -> planner bridge of the reference's cloud node
        (cloud/main_improved_threelayer.py:381-398): occupied sample points of the local grid
        (occupancy > threshold), every `len // max_spheres`-th one becomes a sphere obstacle."""
        grid, occ = self.get_local_occupancy_grid(center, size)
        pts = grid[occ > threshold]
        if pts.size == 0:
            return []
        step = max(1, pts.shape[0] // max_spheres)
        return [(p.copy(), float(radius)) for p in pts[::step]]

    def _sq_scratch(self):
        torch = _torch()
        n = 2 * self.nx * self.ny * self.nz
        if getattr(self, "_sq", None) is None or self._sq.numel() != n:
            self._sq = torch.empty(n, dtype=torch.int32, device=self.device)
        return self._sq

    def signed_distance(self, threshold: float = 0.6, stream=None):
        """Signed distance to the occupied cells (occupancy > threshold), in metres: (nz, ny, nx)
        float32 device tensor, positive in free space, negative inside obstacles, from the exact
        Euclidean distance transform between cell centres (three launches).  With no occupied cell
        every entry is the box diagonal, with no free cell its negative (header:
        dart_map_signed_distance).  Recompute after the map changes."""
        torch = _torch()
        phi = torch.empty((self.nz, self.ny, self.nx), dtype=torch.float32, device=self.device)
        g = self._grid()
        rc = _cabi.lib().dart_map_signed_distance(C.byref(g), float(threshold), phi.data_ptr(),
                                                  self._sq_scratch().data_ptr(), self._stream(stream))
        _cabi.check(rc, "dart_map_signed_distance")
        return phi

    def squared_distance_voxels(self):
        """(nz, ny, nx) int32 view of the exact squared voxel distances the last `signed_distance` /
        `clearance_field` call computed: D+ at free cells, -D- at occupied cells."""
        if getattr(self, "_sq", None) is None:
            raise ValueError("no distance transform has been computed on this grid")
        return self._sq[: self.nx * self.ny * self.nz].view(self.nz, self.ny, self.nx)

    def clearance_field(self, safety_distance: float, threshold: float = 0.6, stream=None) -> "DenseOccupancyGrid":
        """A grid of the same geometry and cell type whose cells are
        ``0.5 + max(0, safety_distance - phi)`` (phi = ``signed_distance(threshold)``) and whose prior
        is 0.5.  As the penalty grid of ``plan_batch(..., obstacle_penalty=True)`` or of
        ``ClosedLoopSim(penalty_grid=...)`` it costs nothing farther than ``safety_distance`` from
        every obstacle and, unlike the occupancy itself, keeps a gradient inside obstacles."""
        torch = _torch()
        out = DenseOccupancyGrid.__new__(DenseOccupancyGrid)
        out.__dict__.update({k: v for k, v in self.__dict__.items() if k not in ("occ", "_counts", "_sq", "_updated")})
        out._counts, out._sq = None, None
        out.prob_prior = 0.5
        out.total_observations = 0
        out.occ = torch.empty_like(self.occ)
        g = self._grid()
        rc = _cabi.lib().dart_map_clearance_field(C.byref(g), float(threshold), float(safety_distance),
                                                  out.prob_prior, out.occ.data_ptr(),
                                                  self._sq_scratch().data_ptr(), self._stream(stream))
        _cabi.check(rc, "dart_map_clearance_field")
        return out

    def get_mapping_stats(self) -> Dict[str, Any]:
        """:353-363 (total_voxels = cells that left the prior)"""
        nvox = int((self.occ != self.prob_prior).sum().item())
        return {"total_voxels": nvox, "total_observations": self.total_observations,
                "memory_efficiency": f"{self.occ.numel() * 4} bytes", "last_update": getattr(self, "last_update_time", 0.0),
                "resolution": self.resolution, "max_range": self.max_range}

    def trace_rays(self, starts, directions, distances, max_vox: int = 0, stream=None):
        """_trace_ray (:250-309) for B rays.  Returns (count (B,) int32, voxels (max_vox,3,B) int32
        or None): voxels[:count[b], :, b] is the reference's list for ray b."""
        torch = _torch()
        s, d = self._soa(starts, 3), self._soa(directions, 3)
        B = s.shape[1]
        dist = torch.as_tensor(np.asarray(distances, np.float64) if not torch.is_tensor(distances) else distances,
                               dtype=torch.float64).to(self.device).reshape(B).contiguous()
        count = torch.empty(B, dtype=torch.int32, device=self.device)
        vox = torch.zeros((max_vox, 3, B), dtype=torch.int32, device=self.device) if max_vox > 0 else None
        rc = _cabi.lib().dart_map_trace_ray_batch(self.resolution, B, B, s.data_ptr(), d.data_ptr(),
                                                  dist.data_ptr(), int(max_vox), count.data_ptr(),
                                                  None if vox is None else vox.data_ptr(),
                                                  self._stream(stream))
        _cabi.check(rc, "dart_map_trace_ray_batch")
        return count, vox

    def _trace_ray(self, start, direction, distance: float, max_vox: int = 4096):
        """Reference signature: list of voxel-index tuples for one ray."""
        count, vox = self.trace_rays(np.asarray(start, float)[None], np.asarray(direction, float)[None],
                                     [distance], max_vox=max_vox)
        n = int(count[0])
        if n > max_vox:
            raise ValueError(f"ray visits {n} voxels > max_vox={max_vox}")
        v = vox[:n, :, 0].cpu().numpy()
        return [tuple(int(c) for c in row) for row in v]
