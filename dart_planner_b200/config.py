"""SE3MPCConfig (mirror of se3_mpc_planner.py:36-79) and the YAML loader the north star asks
for (planning defaults from config/defaults.yaml, airframe mass from config/airframes.yaml).

Quantities: the reference wraps limits in pint Quantities; its solve only ever uses their SI
magnitudes (SURVEY.md App. E).  Anything with a ``.magnitude`` / ``.to(unit)`` is accepted
and stripped to SI floats here; plain floats are taken as SI.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, fields, replace
from typing import Any, Dict, Optional

from ._cabi import Params

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULTS_YAML = os.path.join(_ROOT, "config", "defaults.yaml")
AIRFRAMES_YAML = os.path.join(_ROOT, "config", "airframes.yaml")

# reference: config/frozen_config.py:86 (control_loop_frequency_hz = 400) through
# common/timing_alignment.py:76-78 -- the planner's dt is ALWAYS 1/control frequency
REFERENCE_CONTROL_FREQUENCY_HZ = 400.0


def to_si(value: Any, unit: Optional[str] = None) -> Any:
    """Strip a pint-like Quantity to its SI magnitude (``ensure_units`` + ``to_float``)."""
    if hasattr(value, "to") and unit is not None and hasattr(value, "magnitude"):
        try:
            value = value.to(unit)
        except Exception as exc:  # pint.DimensionalityError and friends
            raise ValueError(f"cannot convert {value!r} to {unit}") from exc
    if hasattr(value, "magnitude"):
        value = value.magnitude
    return value


@dataclass(frozen=True)
class SE3MPCConfig:
    """Same fields, names and defaults as the reference dataclass (se3_mpc_planner.py:36-79)."""

    prediction_horizon: int = 6
    dt: float = 0.125  # overridden by the timing alignment in SE3MPCPlanner.__init__
    max_velocity: float = 10.0        # m/s
    max_acceleration: float = 15.0    # m/s^2   (dead parameter in the reference solve)
    max_jerk: float = 20.0            # m/s^3   (dead)
    max_thrust: float = 25.0          # N
    min_thrust: float = 2.0           # N
    max_tilt_angle: float = math.pi / 4   # rad
    max_angular_velocity: float = 4.0     # rad/s (dead)
    position_weight: float = 100.0
    velocity_weight: float = 10.0
    acceleration_weight: float = 1.0
    thrust_weight: float = 0.1
    angular_weight: float = 10.0      # dead
    obstacle_weight: float = 1000.0   # dead in the reference solve (constraints never passed)
    safety_margin: float = 1.5        # m
    max_iterations: int = 15
    convergence_tolerance: float = 5e-2

    _UNITS = {"max_velocity": "m/s", "max_acceleration": "m/s^2", "max_jerk": "m/s^3",
              "max_thrust": "N", "min_thrust": "N", "max_tilt_angle": "rad",
              "max_angular_velocity": "rad/s", "safety_margin": "m"}

    def __post_init__(self):
        for f in fields(self):
            v = to_si(getattr(self, f.name), self._UNITS.get(f.name))
            if f.name in ("prediction_horizon", "max_iterations"):
                v = int(v)
            else:
                v = float(v)
            object.__setattr__(self, f.name, v)
        if self.prediction_horizon < 1:
            raise ValueError("prediction_horizon must be >= 1")

    def as_dict(self) -> Dict[str, Any]:
        return {f.name: getattr(self, f.name) for f in fields(self)}


class AttrDict(dict):
    """`planner.config` in the reference is a dict that its tests read as attributes
    (tests/test_se3_mpc_with_mapper.py:42, tests/test_sitl_unit_tests.py:46): support both."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e


def make_params(cfg: SE3MPCConfig, *, mass: float = 1.5, gravity: float = 9.81,
                dt: Optional[float] = None, gradient_mode: int = 0, max_corrections: int = 10,
                max_linesearch: int = 20, max_fun: int = 15000,
                obstacle_free_level: float = 0.5) -> Params:
    """SE3MPCConfig -> the C-ABI parameter block, exactly as the reference feeds SciPy
    (se3_mpc_planner.py:256-268, :378-402)."""
    p = Params()
    p.struct_size = C.sizeof(Params)
    p.horizon = int(cfg.prediction_horizon)
    p.max_iterations = int(cfg.max_iterations)
    p.max_corrections = int(max_corrections)
    p.max_linesearch = int(max_linesearch)
    p.max_fun = int(max_fun)
    p.gradient_mode = int(gradient_mode)
    p.dt = float(cfg.dt if dt is None else dt)
    p.mass = float(mass)
    p.gravity = float(gravity)
    p.pos_bound = 100.0
    p.max_velocity = float(cfg.max_velocity)
    p.tilt_thrust = float(cfg.max_thrust * math.sin(cfg.max_tilt_angle))
    p.min_thrust = float(cfg.min_thrust)
    p.max_thrust = float(cfg.max_thrust)
    p.w_pos = float(cfg.position_weight)
    p.w_vel = float(cfg.velocity_weight)
    p.w_acc = float(cfg.acceleration_weight)
    p.w_thrust = float(cfg.thrust_weight)
    p.gtol = float(cfg.convergence_tolerance)
    p.ftol = float(cfg.convergence_tolerance * 10)
    p.w_obstacle = float(cfg.obstacle_weight)          # only read in gradient_modes 2, 4, 5 and 6
    p.obstacle_free_level = float(obstacle_free_level)
    return p


def _resolve_airframe(table: Dict[str, Any], name: str, _depth: int = 0) -> Dict[str, Any]:
    if name not in table:
        raise KeyError(f"airframe {name!r} not in airframes.yaml (have: {sorted(table)})")
    if _depth > 8:
        raise ValueError("airframes.yaml: `extends` chain too deep")
    entry = dict(table[name] or {})
    base = entry.pop("extends", None)
    if base:
        merged = _resolve_airframe(table, base, _depth + 1)
        merged.update(entry)
        return merged
    return entry


def load_airframe(name: str = "default", path: Optional[str] = None) -> Dict[str, Any]:
    import yaml

    with open(path or AIRFRAMES_YAML) as fh:
        table = yaml.safe_load(fh) or {}
    return _resolve_airframe(table, name)


def load_planner_config(defaults_path: Optional[str] = None, airframe: str = "default",
                        airframes_path: Optional[str] = None, **overrides):
    """Returns ``(SE3MPCConfig, mass_kg)`` from the YAML files.

    `planning:` keys that are SE3MPCConfig fields are applied (horizon, dt, weights, tolerance,
    iteration cap, safety margin); unknown keys raise.  The airframe supplies the mass.
    """
    import yaml

    with open(defaults_path or DEFAULTS_YAML) as fh:
        doc = yaml.safe_load(fh) or {}
    planning = dict(doc.get("planning") or {})
    planning.update(overrides)
    names = {f.name for f in fields(SE3MPCConfig)}
    unknown = sorted(set(planning) - names)
    if unknown:
        raise KeyError(f"unknown planning keys in config: {unknown}")
    cfg = replace(SE3MPCConfig(), **planning)
    af = load_airframe(airframe, airframes_path)
    return cfg, float(af.get("mass", 1.5))
