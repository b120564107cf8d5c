"""Goal producer in front of the batched solve (SURVEY.md 8(f)4): `GlobalMissionPlanner.
get_current_goal` (src/dart_planner/planning/global_mission_planner.py:182-224 and the phase
functions :254-404, :450-460) for B drones at once -- the (B, 3) goals go straight into
`plan_batch` / `BatchWorkspace`, so one node serves many edge drones per step.

Mirrors the reference per drone: the mission phase state machine (TAKEOFF -> NAVIGATION ->
LANDING, EMERGENCY below 0.5 m outside LANDING, checked at the global replanning rate), the 2 m
waypoint-reached rule, the semantic adjustments of the approach ("obstacle": back off by the safety
margin along the line to the drone; "landing_pad": 3 m above the pad, or the drone's altitude if
higher; "doorway": exact height), descent goals of LANDING / EMERGENCY, and the exploration spiral
when no uncertainty region is known.  The neural-scene / uncertainty-field updates the reference
runs inside its global planning step produce no goal (placeholders) and are out of scope
(SURVEY.md 2).  Time is an argument (`now`), not the wall clock, so a run is reproducible.
Host-side NumPy: this is bookkeeping, not the solve.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

TAKEOFF, EXPLORATION, MAPPING, NAVIGATION, LANDING, EMERGENCY = range(6)
PHASE_NAMES = ("takeoff", "exploration", "mapping", "navigation", "landing", "emergency")
_LABEL_CODES = {"obstacle": 1, "landing_pad": 2, "doorway": 3}


@dataclass
class SemanticWaypoint:
    """:32-42"""
    position: np.ndarray
    semantic_label: str = "safe_zone"
    uncertainty: float = 0.0
    priority: int = 1

    def __post_init__(self):
        self.position = np.asarray(getattr(self.position, "magnitude", self.position), dtype=np.float64).reshape(3)


@dataclass
class GlobalMissionConfig:
    """:45-63 (the fields the goal logic reads)"""
    exploration_radius: float = 50.0
    safety_margin: float = 2.0
    global_replan_frequency: float = 1.0


class BatchedMissionGoals:
    """B drones flying the same list of semantic waypoints (each with its own progress).

    >>> goals = BatchedMissionGoals(B, waypoints)
    >>> g = goals.get_current_goals(positions, now=t)      # (B, 3), feeds plan_batch
    """

    def __init__(self, B: int, waypoints: Sequence[SemanticWaypoint] = (), config: Optional[GlobalMissionConfig] = None):
        self.B = int(B)
        self.config = config or GlobalMissionConfig()
        self.phase = np.full(self.B, TAKEOFF, dtype=np.int32)                 # :121
        self.waypoint_index = np.zeros(self.B, dtype=np.int64)
        self.last_global_plan_time = np.zeros(self.B)                         # :174
        self.explored_count = np.zeros(self.B, dtype=np.int64)                # len(explored_regions)
        self.set_mission_waypoints(waypoints)

    def set_mission_waypoints(self, waypoints: Sequence[SemanticWaypoint]):
        """:170-180"""
        self.waypoints = list(waypoints)
        self._wp_pos = np.array([w.position for w in self.waypoints], dtype=np.float64).reshape(-1, 3)
        self._wp_label = np.array([_LABEL_CODES.get(w.semantic_label, 0) for w in self.waypoints], dtype=np.int32)
        self.waypoint_index[:] = 0

    # ------------------------------------------------------------------------------------
    def get_current_goals(self, positions, now: float) -> np.ndarray:
        P = np.asarray(positions, dtype=np.float64).reshape(self.B, 3)
        cfg = self.config
        # global replanning at its own rate (:195-201): only the emergency check changes a goal (:450-458)
        due = (now - self.last_global_plan_time) > 1.0 / cfg.global_replan_frequency
        low = due & (P[:, 2] < 0.5) & (self.phase != LANDING)
        self.phase[low] = EMERGENCY
        self.last_global_plan_time[due] = now
        goal = P.copy()                                                        # default: hold position (:222-224)
        ph = self.phase.copy()                                                 # the phase each drone is dispatched on
        # TAKEOFF (:254-265)
        m = ph == TAKEOFF
        goal[m, 2] = 5.0
        self.phase[m & (P[:, 2] >= 5.0 - 0.5)] = NAVIGATION
        # EXPLORATION without known uncertainty regions: the spiral (:279-293)
        m = ph == EXPLORATION
        if m.any():
            angle = self.explored_count[m] * 0.5
            radius = np.minimum(10.0 + self.explored_count[m] * 2.0, cfg.exploration_radius)
            goal[m, 0] = P[m, 0] + radius * np.cos(angle)
            goal[m, 1] = P[m, 1] + radius * np.sin(angle)
        # NAVIGATION / MAPPING (:295-343)
        m = (ph == NAVIGATION) | (ph == MAPPING)
        nwp = len(self.waypoints)
        if m.any() and nwp > 0:
            idx = np.where(m)[0]
            done = self.waypoint_index[idx] >= nwp                             # :307-310
            self.phase[idx[done]] = LANDING
            idx = idx[~done]
            wp = self._wp_pos[self.waypoint_index[idx]]
            reached = np.sqrt(((P[idx] - wp) ** 2).sum(axis=1)) < 2.0          # :315-319
            self.waypoint_index[idx[reached]] += 1
            finished = self.waypoint_index[idx] >= nwp                         # :326-329
            self.phase[idx[finished]] = LANDING
            idx = idx[~finished]
            goal[idx] = self._semantic_goal(self.waypoint_index[idx], P[idx])
        # LANDING (:345-356), EMERGENCY (:358-363)
        m = ph == LANDING
        goal[m, 2] = np.maximum(0.5, P[m, 2] - 1.0)
        m = ph == EMERGENCY
        goal[m, 2] = np.maximum(0.0, P[m, 2] - 2.0)
        return goal

    def _semantic_goal(self, wi, P):
        """:365-392"""
        base = self._wp_pos[wi].copy()
        lab = self._wp_label[wi]
        m = lab == 1                                                           # obstacle
        if m.any():
            d = P[m] - base[m]
            n = np.sqrt((d ** 2).sum(axis=1))
            ok = n > 0
            step = np.zeros_like(d)
            step[ok] = d[ok] / n[ok, None] * self.config.safety_margin
            base[m] = base[m] + step
        m = lab == 2                                                           # landing pad: from above
        base[m, 2] = np.maximum(base[m, 2] + 3.0, P[m, 2])
        return base                                                            # doorway: exact height (unchanged)

    def phase_names(self) -> List[str]:
        return [PHASE_NAMES[p] for p in self.phase]


def reference_path(waypoints, speed: float, dt: float, T: int):
    """Waypoints -> the per-timestep reference of the tracking modes (gradient_mode 7 / 8:
    ``plan_batch(reference=)``, ``ClosedLoopSim(reference_path=)``).

    waypoints : (W, 3), or (B, W, 3) one polyline per drone
    Sample j = 0 .. T-1 is the point at arc length s_j = min((speed * j) * dt, L) along the polyline
    of length L: on segment i with cum_i <= s_j < cum_{i+1} (zero-length segments are never current),
    P_j = w_i + ((s_j - cum_i) / len_i) (w_{i+1} - w_i), and its velocity is speed along that
    segment, V_j = (speed / len_i) (w_{i+1} - w_i).  Once (speed * j) * dt >= L the end is reached:
    P_j = the last waypoint, V_j = +0.
    Returns (P, V), both (B, T, 3) float64 (B = 1 for a single polyline)."""
    w = np.asarray(waypoints, np.float64)
    if w.ndim == 2:
        w = w[None]
    if w.ndim != 3 or w.shape[2] != 3 or w.shape[1] < 1:
        raise ValueError(f"waypoints must be (W, 3) or (B, W, 3), got {np.shape(waypoints)}")
    if not (speed > 0.0) or not (dt > 0.0) or int(T) < 1:
        raise ValueError("reference_path needs speed > 0, dt > 0 and T >= 1")
    B, W, T = w.shape[0], w.shape[1], int(T)
    d = w[:, 1:] - w[:, :-1]                                   # (B, W-1, 3)
    seg = np.sqrt((d * d).sum(axis=2))                         # (B, W-1)
    cum = np.concatenate([np.zeros((B, 1)), np.cumsum(seg, axis=1)], axis=1)
    s_raw = (float(speed) * np.arange(T)) * float(dt)          # (T,)
    P = np.empty((B, T, 3))
    V = np.zeros((B, T, 3))
    for b in range(B):
        L = cum[b, -1]
        done = s_raw >= L
        P[b, done] = w[b, -1]
        j = np.nonzero(~done)[0]
        if len(j):
            s = s_raw[j]
            i = np.minimum(np.searchsorted(cum[b], s, side="right") - 1, W - 2)
            frac = (s - cum[b, i]) / seg[b, i]
            P[b, j] = w[b, i] + frac[:, None] * d[b, i]
            V[b, j] = (float(speed) / seg[b, i])[:, None] * d[b, i]
    return P, V
