"""Reference paths shared by the CPU and GPU tiers of the tracking modes 7 / 8."""
import numpy as np

from dart_planner_b200.mission import reference_path


def circle_paths(B, T, dt, seed=11):
    """One constant-speed circle per drone (radius 2..5 m, 1.5..3 m/s, either direction, level),
    T samples dt apart; the last sample has velocity +0 (the path stops there)."""
    rng = np.random.default_rng(seed)
    c = np.concatenate([rng.uniform(-10, 10, (B, 2)), rng.uniform(3, 8, (B, 1))], 1)
    r = rng.uniform(2, 5, B)
    w = rng.uniform(1.5, 3.0, B) / r * rng.choice([-1.0, 1.0], B)
    th = rng.uniform(0, 2 * np.pi, B)[:, None] + w[:, None] * (np.arange(T) * dt)[None]
    P = np.stack([c[:, 0:1] + r[:, None] * np.cos(th), c[:, 1:2] + r[:, None] * np.sin(th),
                  np.repeat(c[:, 2:3], T, 1)], 2)
    V = np.stack([-(r * w)[:, None] * np.sin(th), (r * w)[:, None] * np.cos(th), np.zeros((B, T))], 2)
    V[:, -1] = 0.0
    return P, V


def polyline_paths(B, T, dt, seed=12, speed=2.5):
    """Four waypoints per drone, three legs of 1..4 m in random directions, the second leg repeated
    as a zero-length segment, sampled by mission.reference_path at `speed` (the path ends by
    t = 4.8 s)."""
    rng = np.random.default_rng(seed)
    d = rng.normal(0, 1, (B, 3, 3))
    d *= (rng.uniform(1, 4, (B, 3)) / np.linalg.norm(d, axis=2))[..., None]
    w0 = np.concatenate([rng.uniform(-10, 10, (B, 1, 2)), rng.uniform(3, 8, (B, 1, 1))], 2)
    w = np.concatenate([w0, w0 + d.cumsum(1)], 1)
    w = np.concatenate([w[:, :2], w[:, 1:2], w[:, 2:]], 1)
    return reference_path(w, speed, dt, T)


def tracking_error(hist, P):
    """hist (S, B, 3): positions after steps 0..S-1; step s ends at time s+1, whose path sample is
    min(s+1, T-1).  -> per-step distance (S, B)."""
    S, T = hist.shape[0], P.shape[1]
    j = np.minimum(np.arange(S) + 1, T - 1)
    return np.linalg.norm(hist - P[:, j].transpose(1, 0, 2), axis=2)
