/*
 * map_query.cuh -- occupancy-grid lookups shared by the mapper kernels and the solve kernel's
 * fused safety check, and the grid check of every entry that takes a grid.  world_to_voxel = floor(p / res) (explicit_geometric_mapper.py:91-94);
 * keys outside the dense grid read the prior, like the reference's dict miss (:154-169).
 */
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/dart_se3mpc.h"

namespace dartb200 {

/* a grid every entry may read: a dense box, a positive voxel size, float32 or float64 cells */
inline int check_grid(const dart_grid *g)
{
    if (!g || !g->occ || g->nx <= 0 || g->ny <= 0 || g->nz <= 0 || !(g->resolution > 0.0))
        return DART_E_BADARG;
    if (g->cell_bytes != 0 && g->cell_bytes != 4 && g->cell_bytes != 8) return DART_E_BADARG;
    return DART_OK;
}

__device__ __forceinline__ int vox(double p, double res) { return (int)floor(p / res); }

/* cell i of the grid as a double: float32 or float64 storage (dart_grid.cell_bytes) */
__device__ __forceinline__ double grid_cell(const dart_grid &g, long long i)
{
    if (g.cell_bytes == 8) return __ldg(static_cast<const double *>(g.occ) + i);
    return (double)__ldg(static_cast<const float *>(g.occ) + i);
}

__device__ __forceinline__ double grid_at(const dart_grid &g, int kx, int ky, int kz)
{
    const int ix = kx - g.ox, iy = ky - g.oy, iz = kz - g.oz;
    if (ix < 0 || iy < 0 || iz < 0 || ix >= g.nx || iy >= g.ny || iz >= g.nz) return g.prior;
    return grid_cell(g, ((long long)iz * g.ny + iy) * g.nx + ix);
}

__device__ __forceinline__ double query(const dart_grid &g, double x, double y, double z)
{
    return grid_at(g, vox(x, g.resolution), vox(y, g.resolution), vox(z, g.resolution));
}

/* is_trajectory_safe's per-position test (:195-219, stencil :338-351): centre, then
 * -x,+x,-y,+y,-z,+z at `margin`; strict `>` like is_collision (:184-193) */
__device__ __forceinline__ bool position_collides(const dart_grid &g, double cx, double cy, double cz,
                                                  double margin, double thr)
{
    const double c[3] = {cx, cy, cz};
    bool col = query(g, c[0], c[1], c[2]) > thr;
#pragma unroll
    for (int axis = 0; axis < 3; ++axis)
#pragma unroll
        for (int dir = -1; dir <= 1; dir += 2) {
            double q[3] = {c[0], c[1], c[2]};
            q[axis] = c[axis] + (double)dir * margin;
            col = col || (query(g, q[0], q[1], q[2]) > thr);
        }
    return col;
}

} /* namespace dartb200 */
