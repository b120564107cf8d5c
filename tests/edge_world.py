"""The grid-edge world of the penalty tests (tests/test_exact_check.py, tests/test_gpu_kernel_matrix.py):
a small occupancy grid with an asymmetric origin and a prior above the free level, and inputs whose
horizons cross its faces and corners."""
import numpy as np

import exact_check as xc

# The grid-edge world: an asymmetric origin, a grid small enough that horizons leave it, and a
# prior above the free level, so that every position outside the grid is penalised.
EDGE_SHAPE = (40, 32, 24)              # nx, ny, nz
EDGE_ORIGIN = (-37, 5, -3)
EDGE_RES = 0.4
EDGE_PRIOR = 0.62
EDGE_FREE = 0.5
EDGE_W = 1000.0


def edge_box():
    lo = np.array(EDGE_ORIGIN, np.float64) * EDGE_RES
    return lo, lo + np.array(EDGE_SHAPE) * EDGE_RES


def edge_cells(dtype, seed=5):
    """(nz, ny, nx) cells: a free background below the free level with a smooth ripple and six
    occupied spheres.  float64 cells carry values float32 cannot hold."""
    nx, ny, nz = EDGE_SHAPE
    ctr = [(np.arange(n) + o + 0.5) * EDGE_RES for n, o in zip(EDGE_SHAPE, EDGE_ORIGIN)]
    Z, Y, X = np.meshgrid(ctr[2], ctr[1], ctr[0], indexing="ij")
    occ = 0.2 + 0.1 * np.sin(0.7 * X + 0.3) * np.cos(0.5 * Y) + 1e-3 * np.sin(1.3 * Z)
    rng = np.random.default_rng(seed)
    lo, hi = edge_box()
    for _ in range(6):
        c, r = rng.uniform(lo + 1, hi - 1), rng.uniform(1.0, 2.5)
        inside = (X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2 <= r * r
        occ[inside] = 0.9 + 0.01 * np.sin(X[inside] * 7.1)
    return np.ascontiguousarray(occ.astype(dtype))


def edge_inputs(B, seed, at_goal=True):
    """Starts inside the grid near its faces and corners, goals across them (some outside), a third
    of the goal coordinates exactly on voxel-centre planes ((k + 1/2) res: interpolation weight 0)."""
    rng = np.random.default_rng(seed)
    lo, hi = edge_box()
    corner = np.where(rng.random((B, 3)) < 0.5, lo, hi)
    p0 = np.where(rng.random((B, 3)) < 0.6, corner + np.sign((lo + hi) / 2 - corner) * rng.uniform(0.2, 2.0, (B, 3)),
                  rng.uniform(lo + 0.5, hi - 0.5, (B, 3)))
    goal = p0 + rng.normal(0, 3.0, (B, 3)) + np.sign(corner - p0) * 1.5
    on_plane = rng.random((B, 3)) < 1 / 3
    goal[on_plane] = (np.floor(goal[on_plane] / EDGE_RES - 0.5) + 0.5) * EDGE_RES
    v0 = rng.uniform(-1.5, 1.5, (B, 3))
    if at_goal:
        p0[::8], v0[::8] = goal[::8], 0.0      # at the goal: stops on the projected gradient
    return p0, v0, goal


def stationary_warm(xw, goal, N, min_thrust=2.0):
    """Warm starts at the stationary point of the reference's gradient for every eighth problem
    (P = goal, V = 0, T = (0, 0, min_thrust)): modes 0 and 2 stop there on the projected gradient."""
    xw = xw.copy()
    xw[::8, :3 * N] = np.tile(goal[::8], (1, N))
    xw[::8, 3 * N:] = 0.0
    xw[::8, 6 * N + 2::3] = min_thrust
    return xw


def oracle_grid(oracle_mod, cells, origin=EDGE_ORIGIN):
    return oracle_mod.DenseGrid.from_cells(cells, origin, EDGE_RES, EDGE_PRIOR)


def exact_grid(cells, origin=EDGE_ORIGIN):
    return xc.Grid(cells, origin, EDGE_RES, EDGE_PRIOR)
