"""Obstacle-aware closed loop, CPU tier: a NumPy/SciPy restatement of the signed distance and the
clearance field (dart_map_signed_distance / dart_map_clearance_field), of the collision sampling of
the closed-loop step with a map (dart_se3mpc_closed_loop_step_map), and the oracle's closed loop in
the two scenarios DESIGN.md 5d reports: the clearance field steers every drone around the
obstacles that the plain dynamics-consistent mode flies through."""
import numpy as np
import pytest
from scipy import ndimage

import rollout_oracle

from test_rollout_mode import GOAL_RADIUS, _world

FREE_LEVEL = 0.5
MAX_SAMPLES = 64


# ---- restatement of the device transform ---------------------------------------------------------
def squared_distances(occ, threshold):
    """(D+, D-) exact integer squared voxel distances between cell centres: D+ to the nearest
    occupied cell (occ > threshold), D- to the nearest free one; the squared box diagonal where
    there is no such cell."""
    o = np.asarray(occ).astype(np.float64) > threshold
    diag2 = sum(s * s for s in o.shape)

    def to_sites(sites):
        if not sites.any():
            return np.full(o.shape, diag2, np.int64)
        _, idx = ndimage.distance_transform_edt(~sites, return_indices=True)
        grid = np.indices(o.shape)
        return ((idx - grid) ** 2).sum(axis=0).astype(np.int64)

    return to_sites(o), to_sites(~o)


def signed_distance(occ, res, threshold):
    """phi = res (sqrt(D+) - sqrt(D-)) in float64, rounded once to float32."""
    dp, dm = squared_distances(occ, threshold)
    return (res * (np.sqrt(dp.astype(np.float64)) - np.sqrt(dm.astype(np.float64)))).astype(np.float32)


def clearance_field(occ, res, threshold, safety_distance, free_level=FREE_LEVEL):
    """c = free_level + max(0, d_safe - phi), in the cell type of the source grid."""
    phi = signed_distance(occ, res, threshold).astype(np.float64)
    return (free_level + np.maximum(0.0, safety_distance - phi)).astype(np.asarray(occ).dtype)


def signed_squared(occ, threshold):
    """What the device leaves in its scratch: D+ at free cells, -D- at occupied cells."""
    dp, dm = squared_distances(occ, threshold)
    return np.where(dm > 0, -dm, dp)


# ---- restatement of the closed loop's collision sampling ------------------------------------------
def query(occ, origin, res, prior, q):
    """floor(q / res) keys, the prior outside the box (map_query.cuh)."""
    k = [np.floor(q[:, c] / res).astype(np.int64) - origin[c] for c in range(3)]
    nz, ny, nx = occ.shape
    inside = (k[0] >= 0) & (k[0] < nx) & (k[1] >= 0) & (k[1] < ny) & (k[2] >= 0) & (k[2] < nz)
    val = np.full(q.shape[0], float(prior))
    val[inside] = np.asarray(occ)[k[2][inside], k[1][inside], k[0][inside]].astype(np.float64)
    return val


def collides(occ, origin, res, prior, q, margin, threshold):
    """is_trajectory_safe's per-position stencil: centre, then -x,+x,-y,+y,-z,+z at margin."""
    col = query(occ, origin, res, prior, q) > threshold
    for axis in range(3):
        for d in (-1.0, 1.0):
            qq = q.copy()
            qq[:, axis] = q[:, axis] + d * margin
            col |= query(occ, origin, res, prior, qq) > threshold
    return col


def path_collides(occ, origin, res, prior, p, pn, margin, threshold):
    """The plant's path of one step, p -> pn, at q_j = p + (pn - p)(j / S), j = 1..S,
    S = max(1, ceil(|pn - p|_inf / (res / 2))) capped at 64."""
    d = pn - p
    m = np.abs(d).max(axis=1)
    h = 0.5 * res
    with np.errstate(invalid="ignore"):
        S = np.where(m <= MAX_SAMPLES * h, np.maximum(1.0, np.ceil(m / h)), MAX_SAMPLES).astype(np.int64)
    hit = np.zeros(p.shape[0], bool)
    for j in range(1, MAX_SAMPLES + 1):
        on = j <= S
        if not on.any():
            break
        q = p[on] + d[on] * (j / S[on])[:, None]
        hit[np.where(on)[0]] |= collides(occ, origin, res, prior, q, margin, threshold)
    return hit


# ---- scenarios ----------------------------------------------------------------------------------
RES, SHAPE, ORIGIN = 0.4, (128, 128, 128), (-64, -64, -64)


def one_sphere(oracle_mod):
    """A sphere of radius 2.5 m at (0, 0, 5); drones fly from x = -12 to x = +12 with lateral
    offsets in +-2 m, straight through it."""
    og = oracle_mod.DenseGrid(SHAPE, ORIGIN, RES)
    og.add_sphere(np.array([0.0, 0.0, 5.0]), 2.5)
    B = 128
    off = np.random.default_rng(3).uniform(-2, 2, (B, 2))
    p0 = np.stack([np.full(B, -12.0), off[:, 0], 5 + off[:, 1]], 1)
    goal = np.stack([np.full(B, 12.0), off[:, 0], 5 + off[:, 1]], 1)
    return og, p0, goal


def sphere_world(oracle_mod, B=256, threshold=0.6, clearance=1.5, seed=4):
    """The 48-sphere world of test_rollout_mode; configs[4]-like starts and goals at least
    `clearance` m from every occupied cell."""
    og = _world(oracle_mod)
    phi = signed_distance(og.occ, RES, threshold)

    def phi_at(p):
        k = np.floor(p / RES).astype(int) - np.array(ORIGIN)
        return phi[k[:, 2], k[:, 1], k[:, 0]]

    rng = np.random.default_rng(seed)
    p0 = rng.uniform(-10, 10, (4 * B, 3))
    goal = np.concatenate([rng.uniform(-15, 15, (4 * B, 2)), rng.uniform(3, 8, (4 * B, 1))], 1)
    ok = (phi_at(p0) > clearance) & (phi_at(goal) > clearance)
    assert ok.sum() >= B
    return og, p0[ok][:B], goal[ok][:B]


def field_grid(oracle_mod, og, safety_distance, threshold=0.6):
    fg = oracle_mod.DenseGrid(SHAPE, ORIGIN, RES, prior=FREE_LEVEL)
    fg.occ[...] = clearance_field(og.occ, RES, threshold, safety_distance)
    return fg


def oracle_loop(oracle_mod, og, p0, goal, penalty=None, weight=0.0, steps=100, N=8, dt=0.1, tol=1e-3):
    """The oracle's closed loop (plant state = the plan's P_1 / V_1) with the flown path of every
    step checked against og (margin 0, threshold 0.6) -> (first collision step, final positions)."""
    op = oracle_mod.make_params(horizon=N, dt=dt, convergence_tolerance=tol)
    kw = dict(grid=penalty, obstacle_weight=weight, free_level=FREE_LEVEL) if penalty is not None else {}
    p, v, x = p0.copy(), np.zeros_like(p0), None
    first = np.full(len(p0), -1)
    for s in range(steps):
        x = rollout_oracle.solve_batch(op, p, v, goal, x_warm=x, nthreads=16, **kw).x
        pn, v = x[:, 3:6].copy(), x[:, 3 * N + 3:3 * N + 6].copy()
        hit = path_collides(og.occ, ORIGIN, RES, og.g.prior, p, pn, 0.0, 0.6)
        first[hit & (first < 0)] = s
        p = pn
    return first, p


# ---- tests --------------------------------------------------------------------------------------
def _brute_force(occ, threshold):
    o = occ.astype(np.float64) > threshold
    cells = np.argwhere(np.ones(o.shape, bool))
    diag2 = sum(s * s for s in o.shape)

    def to(sites):
        pts = np.argwhere(sites)
        if len(pts) == 0:
            return np.full(o.shape, diag2)
        return ((cells[:, None, :] - pts[None]) ** 2).sum(-1).min(1).reshape(o.shape)

    return to(o), to(~o)


@pytest.mark.parametrize("shape", [(5, 7, 9), (1, 1, 13), (6, 1, 4)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_restatement_matches_brute_force(shape, dtype):
    rng = np.random.default_rng(sum(shape))
    for frac in (0.0, 0.1, 0.5, 1.0):
        occ = np.where(rng.random(shape) < frac, 0.9, 0.3).astype(dtype)
        dp, dm = squared_distances(occ, 0.6)
        bp, bm = _brute_force(occ, 0.6)
        np.testing.assert_array_equal(dp, bp)
        np.testing.assert_array_equal(dm, bm)


def test_signed_distance_edge_cases():
    res = 0.25
    # one-voxel-thick wall at x = 4: the distance grows linearly on both sides, -1 voxel inside
    occ = np.full((3, 4, 10), 0.5, np.float32)
    occ[:, :, 4] = 0.9
    phi = signed_distance(occ, res, 0.6)
    np.testing.assert_array_equal(phi[1, 2], np.array([4, 3, 2, 1, -1, 1, 2, 3, 4, 5], np.float32) * res)
    # empty and full grids: plus / minus the box diagonal
    diag = np.float32(res * np.sqrt(3 * 3 + 4 * 4 + 10 * 10))
    assert (signed_distance(np.full((3, 4, 10), 0.5), res, 0.6) == diag).all()
    assert (signed_distance(np.full((3, 4, 10), 0.9), res, 0.6) == -diag).all()
    # a cell exactly at the threshold is free (strict test); float64 cells keep the exact value
    occ = np.full((1, 1, 5), 0.5)
    occ[0, 0, 2] = 0.6
    assert (signed_distance(occ, res, 0.6) == np.float32(res * np.sqrt(1 + 1 + 25))).all()
    occ[0, 0, 2] = np.nextafter(0.6, 1.0)
    wall = np.array([2.0, 1.0, -1.0, 1.0, 2.0]) * res
    np.testing.assert_array_equal(signed_distance(occ, res, 0.6)[0, 0], wall.astype(np.float32))
    # the clearance field: free_level beyond d_safe, rising into the obstacle, in the source type
    f = clearance_field(occ, res, 0.6, 0.3)
    assert f.dtype == np.float64
    np.testing.assert_array_equal(f[0, 0], 0.5 + np.maximum(0.0, 0.3 - wall))
    assert f[0, 0, 0] == 0.5 and f[0, 0, 2] > f[0, 0, 1] > 0.5


def test_path_sampling_restatement():
    occ = np.full((1, 1, 10), 0.5, np.float32)
    occ[0, 0, 5] = 0.9
    p = np.array([[0.05, 0.05, 0.05], [0.05, 0.05, 0.05], [0.05, 0.05, 0.05]])
    pn = np.array([[0.95, 0.05, 0.05], [0.45, 0.05, 0.05], [0.95, 0.05, 0.05]])
    hit = path_collides(occ, (0, 0, 0), 0.1, 0.5, p, pn, 0.0, 0.6)
    assert hit.tolist() == [True, False, True]     # the wall cell lies on the first and third path
    assert not path_collides(occ, (0, 0, 0), 0.1, 0.5, p[:1], p[:1], 0.0, 0.6)[0]


def test_oracle_loop_one_sphere(oracle_mod):
    """Mode 3 flies (almost) every drone through the sphere; the 1 m clearance field at weight 1e5
    steers every one around it, and every drone still ends at its goal."""
    og, p0, goal = one_sphere(oracle_mod)
    first3, _ = oracle_loop(oracle_mod, og, p0, goal)
    assert (first3 >= 0).mean() >= 0.9
    first4, p = oracle_loop(oracle_mod, og, p0, goal, penalty=field_grid(oracle_mod, og, 1.0), weight=1e5)
    assert (first4 < 0).all()
    assert np.linalg.norm(p - goal, axis=1).max() <= GOAL_RADIUS


def test_oracle_loop_sphere_world(oracle_mod):
    og, p0, goal = sphere_world(oracle_mod)
    first3, _ = oracle_loop(oracle_mod, og, p0, goal)
    assert (first3 >= 0).mean() >= 0.05
    first4, p = oracle_loop(oracle_mod, og, p0, goal, penalty=field_grid(oracle_mod, og, 1.0), weight=1e5)
    assert (first4 < 0).all()
    assert np.linalg.norm(p - goal, axis=1).max() <= GOAL_RADIUS
