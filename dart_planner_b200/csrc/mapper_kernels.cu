/*
 * mapper_kernels.cu -- occupancy-map queries next to the solve path, on a dense device grid.
 * Replaces (batched): ExplicitGeometricMapper.query_occupancy_batch / is_trajectory_safe /
 * _trace_ray / add_obstacle (perception/explicit_geometric_mapper.py:154-219, 250-309,
 * 338-351, 399-423).  Integer results are bit-exact with the reference: the file is compiled
 * with -fmad=false so floor(p/res), the DDA distances and the sphere test round exactly like
 * NumPy's separate multiply/add.
 *
 * These are gather kernels (HBM/L2 latency bound): one thread per query / trajectory / ray,
 * batch-major SoA inputs so a warp's loads of each coordinate row are coalesced.  The grid
 * (64 MiB at 256^3 fp32) fits the 126 MB L2, but a query kernel also streams its own inputs and
 * outputs through it (32 B per query, as many sectors as the gathers) and the first touch of every
 * grid sector misses: one cold launch of 4 Mi random queries measures 24 % L2 hits under ncu
 * (which flushes the caches before the launch) -- about half of the gathers hit, none of the
 * streamed sectors; profiles/README.md, round 2.
 */
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/dart_se3mpc.h"
#include "map_query.cuh"

using namespace dartb200;

extern "C" void dart_count_launch_(void);

namespace {

__global__ void __launch_bounds__(256)
map_query_kernel(const __grid_constant__ dart_grid g, long long B, long long ld, const double *pos,
                 double *out)
{
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x)
        out[b] = query(g, __ldg(pos + b), __ldg(pos + ld + b), __ldg(pos + 2 * ld + b));
}

/* is_trajectory_safe: centre, then -x,+x,-y,+y,-z,+z at `margin`; first colliding index */
__global__ void __launch_bounds__(256)
map_traj_safe_kernel(const __grid_constant__ dart_grid g, long long B, long long ld, int npos,
                     const double *pos, double margin, double thr, int *first_hit)
{
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x) {
        int hit = -1;
        for (int i = 0; i < npos && hit < 0; ++i) {
            const double c[3] = {__ldg(pos + (long long)(3 * i) * ld + b),
                                 __ldg(pos + (long long)(3 * i + 1) * ld + b),
                                 __ldg(pos + (long long)(3 * i + 2) * ld + b)};
            const bool col = position_collides(g, c[0], c[1], c[2], margin, thr);
            if (col) hit = i;
        }
        first_hit[b] = hit;
    }
}

/* _trace_ray: Amanatides-Woo DDA with the reference's quirks (step from voxel indices,
 * tie -> lowest axis, loop while cur != end and total <= dist).  visit(kx, ky, kz, n) is called
 * for every voxel in order (n = index along the ray); returns the number of voxels. */
template <class Visit>
__device__ __forceinline__ int dda_walk(double res, const double s[3], const double d_in[3],
                                        double distance, Visit &&visit)
{
    double d[3], tdelta[3], tmax[3];
    int cur[3], endv[3], step[3];
    const double nrm = sqrt((d_in[0] * d_in[0] + d_in[1] * d_in[1]) + d_in[2] * d_in[2]);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        d[c] = d_in[c] / nrm;
        const double e = s[c] + d[c] * distance;
        cur[c] = vox(s[c], res);
        endv[c] = vox(e, res);
    }
    int n = 0;
    visit(cur[0], cur[1], cur[2], n);
    ++n;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        step[c] = endv[c] > cur[c] ? 1 : (endv[c] < cur[c] ? -1 : 0);
        if (step[c] != 0) {
            tdelta[c] = res / fabs(d[c]);
            const double boundary = (double)(cur[c] + (step[c] > 0 ? 1 : 0)) * res;
            tmax[c] = fabs((boundary - s[c]) / d[c]);
        } else {
            tdelta[c] = INFINITY;
            tmax[c] = INFINITY;
        }
    }
    double total = 0.0;
    while ((cur[0] != endv[0] || cur[1] != endv[1] || cur[2] != endv[2]) && total <= distance) {
        int axis = 0;
        if (tmax[1] < tmax[axis]) axis = 1;
        if (tmax[2] < tmax[axis]) axis = 2;
        /* register-friendly select instead of dynamic indexing */
        if (axis == 0) {
            cur[0] += step[0]; total = tmax[0]; tmax[0] += tdelta[0];
        } else if (axis == 1) {
            cur[1] += step[1]; total = tmax[1]; tmax[1] += tdelta[1];
        } else {
            cur[2] += step[2]; total = tmax[2]; tmax[2] += tdelta[2];
        }
        visit(cur[0], cur[1], cur[2], n);
        ++n;
        if (n > (1 << 24)) break; /* NaN guard */
    }
    return n;
}

__global__ void __launch_bounds__(256)
map_trace_ray_kernel(double res, long long B, long long ld, const double *start, const double *dir,
                     const double *dist, int max_vox, int *count, int *voxels)
{
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x) {
        double s[3], d[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            s[c] = __ldg(start + c * ld + b);
            d[c] = __ldg(dir + c * ld + b);
        }
        count[b] = dda_walk(res, s, d, __ldg(dist + b), [&](int kx, int ky, int kz, int n) {
            if (voxels && n < max_vox) {
                int *v = voxels + ((long long)n * 3) * ld + b;
                v[0] = kx;
                v[ld] = ky;
                v[2 * ld] = kz;
            }
        });
    }
}

/* update_map (:100-152), pass 1: one thread per observation walks its ray and COUNTS the visits
 * per voxel (misses in the low word, endpoint hits in the high word of a 64-bit counter) with
 * atomics -- integer, hence independent of the order rays are processed in.  Pass 2 applies
 * the Bayes rule (:311-336) that many times.  The reference applies the same updates in
 * observation order; both likelihoods raise the odds (the reference's miss likelihood is
 * 1 - prob_miss = 0.6, SURVEY App. D) and the clip at 0.99 is a fixed point, so the result is
 * order-independent up to rounding. */
__global__ void __launch_bounds__(256)
map_update_rays_kernel(const __grid_constant__ dart_grid g, long long B, long long ld,
                       const double *start, const double *dir, const double *hit,
                       const double *obs_max_range, double mapper_max_range,
                       unsigned long long *counts, unsigned long long *updated_total)
{
    long long visits = 0;
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x) {
        double s[3], d[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            s[c] = __ldg(start + c * ld + b);
            d[c] = __ldg(dir + c * ld + b);
        }
        const double h = __ldg(hit + b);
        const bool none = isnan(h);
        double hd = (none || h == 0.0) ? __ldg(obs_max_range + b) : h; /* falsy -> max_range (:112) */
        hd = fmin(hd, mapper_max_range);
        /* the last voxel is only known when the walk ends: count every voxel as a miss, then
         * move the last one to the hit word if the observation had a return */
        long long last = -1;
        const int n = dda_walk(g.resolution, s, d, hd, [&](int kx, int ky, int kz, int) {
            const int ix = kx - g.ox, iy = ky - g.oy, iz = kz - g.oz;
            last = -1;
            if (ix < 0 || iy < 0 || iz < 0 || ix >= g.nx || iy >= g.ny || iz >= g.nz) return;
            last = ((long long)iz * g.ny + iy) * g.nx + ix;
            atomicAdd(counts + last, 1ull);
        });
        if (!none && last >= 0) atomicAdd(counts + last, (1ull << 32) - 1ull); /* -1 miss, +1 hit */
        visits += n;
    }
    /* block-level sum of the visit counter, one atomic per warp */
    for (int o = 16; o > 0; o >>= 1) visits += __shfl_xor_sync(0xffffffffu, visits, o);
    if ((threadIdx.x & 31) == 0 && updated_total && visits) atomicAdd(updated_total, (unsigned long long)visits);
}

__device__ __forceinline__ double bayes_update(double p, double lik)
{
    const double num = lik * p;
    const double den = lik * p + (1.0 - lik) * (1.0 - p);
    if (den > 0.0) p = num / den;
    return fmin(fmax(p, 0.01), 0.99);
}

template <class CELL>
__device__ __forceinline__ void apply_cell(CELL *occ, unsigned long long *counts, long long i,
                                           unsigned long long c, double lik_hit, double lik_miss)
{
    counts[i] = 0ull; /* leave the scratch zeroed for the next scan */
    unsigned miss = (unsigned)(c & 0xffffffffull), hitn = (unsigned)(c >> 32);
    double p = (double)occ[i];
    /* 0.99 is a fixed point of both updates after the clip: 64 applications saturate */
    if (miss > 64u) miss = 64u;
    if (hitn > 64u) hitn = 64u;
    /* an update that leaves p unchanged (the clip's fixed point) makes the rest of its run a
     * no-op: stop there -- same result, ~12 instead of up to 64 updates per run */
    for (unsigned k = 0; k < miss; ++k) {
        const double pn = bayes_update(p, lik_miss);
        if (pn == p) break;
        p = pn;
    }
    for (unsigned k = 0; k < hitn; ++k) {
        const double pn = bayes_update(p, lik_hit);
        if (pn == p) break;
        p = pn;
    }
    occ[i] = (CELL)p;
}

/* pass 2: a streaming read of the 8-byte counters (four cells = two 16-byte loads per thread and
 * trip, so enough bytes are in flight to cover the HBM latency); untouched cells cost nothing more */
template <class CELL>
__global__ void __launch_bounds__(256)
map_apply_counts_kernel(CELL *occ, unsigned long long *counts, long long ncell, double lik_hit,
                        double lik_miss)
{
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthr = (long long)gridDim.x * blockDim.x;
    const bool aligned = (reinterpret_cast<unsigned long long>(counts) & 15ull) == 0ull;
    const long long n4 = aligned ? ncell / 4 : 0;
    const ulonglong2 *c2 = reinterpret_cast<const ulonglong2 *>(counts);
    for (long long q = tid; q < n4; q += nthr) {
        const ulonglong2 a = c2[2 * q], b = c2[2 * q + 1];
        if ((a.x | a.y | b.x | b.y) == 0ull) continue;
        if (a.x) apply_cell(occ, counts, 4 * q, a.x, lik_hit, lik_miss);
        if (a.y) apply_cell(occ, counts, 4 * q + 1, a.y, lik_hit, lik_miss);
        if (b.x) apply_cell(occ, counts, 4 * q + 2, b.x, lik_hit, lik_miss);
        if (b.y) apply_cell(occ, counts, 4 * q + 3, b.y, lik_hit, lik_miss);
    }
    for (long long i = 4 * n4 + tid; i < ncell; i += nthr) {
        const unsigned long long c = counts[i];
        if (c) apply_cell(occ, counts, i, c, lik_hit, lik_miss);
    }
}

/* add_obstacle: one block per sphere, threads sweep the (2r+1)^3 cube; voxel CORNER distance */
template <class CELL>
__global__ void __launch_bounds__(256)
map_add_spheres_kernel(const __grid_constant__ dart_grid g, CELL *occ, int nsph,
                       const double *centers, const double *radii, CELL value)
{
    const int sidx = blockIdx.x;
    if (sidx >= nsph) return;
    const double cx = centers[sidx], cy = centers[nsph + sidx], cz = centers[2 * nsph + sidx];
    const double rad = radii[sidx];
    const int vcx = vox(cx, g.resolution), vcy = vox(cy, g.resolution), vcz = vox(cz, g.resolution);
    const int vr = (int)ceil(rad / g.resolution);
    const int w = 2 * vr + 1;
    const long long total = (long long)w * w * w;
    for (long long t = threadIdx.x; t < total; t += blockDim.x) {
        const int dz = (int)(t % w) - vr, dy = (int)((t / w) % w) - vr, dx = (int)(t / ((long long)w * w)) - vr;
        const int kx = vcx + dx, ky = vcy + dy, kz = vcz + dz;
        const double wx = (double)kx * g.resolution - cx, wy = (double)ky * g.resolution - cy,
                     wz = (double)kz * g.resolution - cz;
        const double dist = sqrt((wx * wx + wy * wy) + wz * wz);
        if (dist <= rad) {
            const int ix = kx - g.ox, iy = ky - g.oy, iz = kz - g.oz;
            if (ix < 0 || iy < 0 || iz < 0 || ix >= g.nx || iy >= g.ny || iz >= g.nz) continue;
            occ[((long long)iz * g.ny + iy) * g.nx + ix] = value;
        }
    }
}

/* Exact Euclidean distance transform of the occupancy (`occ > threshold`, is_collision's strict
 * test) for the signed distance and the clearance field: the separable lower envelope of parabolas
 * of Felzenszwalb & Huttenlocher ("Distance Transforms of Sampled Functions", Theory of Computing
 * 8, 2012), one pass along x, y, z, every comparison in integers (no intersection is ever formed
 * as a float).  Between passes a cell is ONE int32: +D at a free cell (squared voxel distance to
 * the nearest occupied cell found so far) and -D at an occupied cell (to the nearest free cell).
 * The other distance of a cell is 0 at every stage -- the cell is a site of that transform -- so
 * the sign says which transform the magnitude belongs to.  EDT_INF: no site on the lines so far.
 * One thread per line; its envelope (sites and f(q) + q^2) lives in shared memory. */
constexpr int EDT_INF = 0x3fffffff;

template <bool FROM_GRID, bool LAST, class CELL>
__global__ void __launch_bounds__(32)
map_edt_pass_kernel(const __grid_constant__ dart_grid g, double thr, int axis, const int *src, int *dst,
                    float *phi, CELL *field, double dsafe, double free_level, int diag2)
{
    extern __shared__ int edt_env[];
    const int T = blockDim.x, t = threadIdx.x;
    const int n = axis == 0 ? g.nx : (axis == 1 ? g.ny : g.nz);
    const long long stride = axis == 0 ? 1ll : (axis == 1 ? (long long)g.nx : (long long)g.nx * g.ny);
    const long long nlines = (long long)g.nx * g.ny * g.nz / n;
    const long long line = (long long)blockIdx.x * T + t;
    if (line >= nlines) return;
    /* lines of one block are neighbours in x (y and z passes: coalesced) or in y (x pass) */
    const long long base = axis == 0 ? line * g.nx
                         : (axis == 1 ? (line / g.nx) * ((long long)g.nx * g.ny) + line % g.nx : line);
    auto enc = [&](int q) -> int {
        const long long i = base + q * stride;
        if constexpr (FROM_GRID) {
            const double o = g.cell_bytes == 8 ? __ldg(static_cast<const double *>(g.occ) + i)
                                               : (double)__ldg(static_cast<const float *>(g.occ) + i);
            return o > thr ? -EDT_INF : EDT_INF;
        } else {
            return __ldg(src + i);
        }
    };
    int *sv = edt_env + t, *sh = edt_env + T + t; /* site k: sv[2kT], sh[2kT] */
#pragma unroll 1
    for (int sgn = 1; sgn >= -1; sgn -= 2) {
        /* lower envelope of f(q) + (p - q)^2 over the sites with f(q) < EDT_INF, f = the sign's
         * distance (0 at the cells of the other sign) */
        int k = -1;
        for (int q = 0; q < n; ++q) {
            const int e = enc(q);
            const int f = sgn > 0 ? max(e, 0) : max(-e, 0);
            if (f >= EDT_INF) continue;
            const long long h = (long long)f + (long long)q * q;
            /* pop while the new parabola's intersection with the top one lies at or left of the
             * top one's intersection with the one below:  (h - ha) / 2(q - a) <= (ha - hb) / 2(a - b) */
            while (k >= 1) {
                const long long a = sv[2 * k * T], b = sv[2 * (k - 1) * T];
                const long long ha = sh[2 * k * T], hb = sh[2 * (k - 1) * T];
                if ((h - ha) * (a - b) <= (ha - hb) * (q - a)) --k;
                else break;
            }
            ++k;
            sv[2 * k * T] = q;
            sh[2 * k * T] = (int)h;
        }
        int j = 0;
        for (int p = 0; p < n; ++p) {
            /* advance while the next parabola's intersection lies left of p */
            while (j < k && (long long)(sh[2 * (j + 1) * T] - sh[2 * j * T]) <
                                2ll * p * (sv[2 * (j + 1) * T] - sv[2 * j * T]))
                ++j;
            const int e = enc(p);
            if ((sgn > 0) != (e > 0)) continue; /* the other transform's cell */
            int D = EDT_INF;
            if (k >= 0) {
                const long long q = sv[2 * j * T];
                D = (int)((long long)sh[2 * j * T] - 2ll * p * q + (long long)p * p);
            }
            const long long i = base + p * stride;
            if constexpr (LAST) {
                /* no site anywhere: the box diagonal (any finite distance is shorter) */
                D = min(D, diag2);
                dst[i] = sgn > 0 ? D : -D;
                const double dp = sgn > 0 ? (double)D : 0.0, dm = sgn > 0 ? 0.0 : (double)D;
                const float ph = (float)(g.resolution * (sqrt(dp) - sqrt(dm)));
                if (phi) phi[i] = ph;
                if (field) field[i] = (CELL)(free_level + fmax(0.0, dsafe - (double)ph));
            } else {
                dst[i] = sgn > 0 ? D : -D;
            }
        }
    }
}

template <bool FROM_GRID, bool LAST, class CELL>
int launch_edt_pass(const dart_grid &g, double thr, int axis, const int *src, int *dst, float *phi,
                    CELL *field, double dsafe, double free_level, int diag2, cudaStream_t s)
{
    const int n = axis == 0 ? g.nx : (axis == 1 ? g.ny : g.nz);
    const long long nlines = (long long)g.nx * g.ny * g.nz / n;
    int T = 49152 / (8 * n);
    T = T < 1 ? 1 : (T > 32 ? 32 : T);
    const int smem = 8 * n * T;
    const void *fn = (const void *)map_edt_pass_kernel<FROM_GRID, LAST, CELL>;
    if (smem > 49152 && cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
        return DART_E_CUDA;
    map_edt_pass_kernel<FROM_GRID, LAST, CELL><<<(unsigned)((nlines + T - 1) / T), T, smem, s>>>(
        g, thr, axis, src, dst, phi, field, dsafe, free_level, diag2);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}

/* the three passes: grid -> S0 (x), S0 -> S1 (y), S1 -> S0 (z, with phi / the field) */
template <class CELL>
int edt(const dart_grid &g, double thr, float *phi, CELL *field, double dsafe, double free_level, int *scratch,
        cudaStream_t s)
{
    const long long ncell = (long long)g.nx * g.ny * g.nz;
    const long long diag2 = (long long)g.nx * g.nx + (long long)g.ny * g.ny + (long long)g.nz * g.nz;
    /* every D and f(q) + q^2 stays below EDT_INF, and a line's envelope fits one block's shared memory */
    if (diag2 >= EDT_INF) return DART_E_UNSUPPORTED;
    int *s0 = scratch, *s1 = scratch + ncell;
    int rc = launch_edt_pass<true, false, CELL>(g, thr, 0, nullptr, s0, nullptr, nullptr, 0.0, 0.0, 0, s);
    if (!rc) rc = launch_edt_pass<false, false, CELL>(g, thr, 1, s0, s1, nullptr, nullptr, 0.0, 0.0, 0, s);
    if (!rc) rc = launch_edt_pass<false, true, CELL>(g, thr, 2, s1, s0, phi, field, dsafe, free_level, (int)diag2, s);
    return rc;
}

int grid_blocks(long long B)
{
    long long nb = (B + 255) / 256;
    const long long cap = 148 * 8;
    return (int)(nb < cap ? (nb < 1 ? 1 : nb) : cap);
}

int check_grid(const dart_grid *g)
{
    if (!g || !g->occ || g->nx <= 0 || g->ny <= 0 || g->nz <= 0 || !(g->resolution > 0.0))
        return DART_E_BADARG;
    if (g->cell_bytes != 0 && g->cell_bytes != 4 && g->cell_bytes != 8) return DART_E_BADARG;
    return DART_OK;
}

} /* namespace */

extern "C" {

int dart_map_query_batch(const dart_grid *g, int64_t B, int64_t ld, const double *pos,
                         double *occ_out, void *stream)
{
    if (check_grid(g) || B < 0 || ld < B || !pos || !occ_out) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    map_query_kernel<<<grid_blocks(B), 256, 0, (cudaStream_t)stream>>>(*g, B, ld, pos, occ_out);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}

int dart_map_traj_safe_batch(const dart_grid *g, int64_t B, int64_t ld, int32_t npos,
                             const double *positions, double margin, double threshold,
                             int32_t *first_hit, void *stream)
{
    if (check_grid(g) || B < 0 || ld < B || npos < 0 || !positions || !first_hit) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    map_traj_safe_kernel<<<grid_blocks(B), 256, 0, (cudaStream_t)stream>>>(*g, B, ld, npos, positions,
                                                                          margin, threshold, first_hit);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}

int dart_map_trace_ray_batch(double resolution, int64_t B, int64_t ld, const double *start,
                             const double *dir, const double *dist, int32_t max_vox,
                             int32_t *count, int32_t *voxels, void *stream)
{
    if (!(resolution > 0.0) || B < 0 || ld < B || !start || !dir || !dist || !count || max_vox < 0)
        return DART_E_BADARG;
    if (B == 0) return DART_OK;
    map_trace_ray_kernel<<<grid_blocks(B), 256, 0, (cudaStream_t)stream>>>(resolution, B, ld, start, dir,
                                                                          dist, max_vox, count, voxels);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}

int dart_map_update_batch(const dart_grid *g, void *occ_writable, uint64_t *counts, int64_t B,
                          int64_t ld, const double *start, const double *dir,
                          const double *hit_distance, const double *obs_max_range,
                          double mapper_max_range, double prob_hit, double prob_miss,
                          uint64_t *updated_voxels, void *stream)
{
    if (check_grid(g) || !occ_writable || !counts || B < 0 || ld < B || !start || !dir || !hit_distance ||
        !obs_max_range || !(mapper_max_range > 0.0))
        return DART_E_BADARG;
    if (B == 0) return DART_OK;
    map_update_rays_kernel<<<grid_blocks(B), 256, 0, (cudaStream_t)stream>>>(
        *g, B, ld, start, dir, hit_distance, obs_max_range, mapper_max_range,
        (unsigned long long *)counts, (unsigned long long *)updated_voxels);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    const long long ncell = (long long)g->nx * g->ny * g->nz;
    /* likelihoods exactly as _bayesian_update forms them (:322-327) */
    if (g->cell_bytes == 8)
        map_apply_counts_kernel<double><<<grid_blocks(ncell), 256, 0, (cudaStream_t)stream>>>(
            (double *)occ_writable, (unsigned long long *)counts, ncell, prob_hit, 1.0 - prob_miss);
    else
        map_apply_counts_kernel<float><<<grid_blocks(ncell), 256, 0, (cudaStream_t)stream>>>(
            (float *)occ_writable, (unsigned long long *)counts, ncell, prob_hit, 1.0 - prob_miss);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}

int dart_map_add_spheres(const dart_grid *g, void *occ_writable, int32_t n, const double *centers,
                         const double *radii, double value, void *stream)
{
    if (check_grid(g) || !occ_writable || n < 0 || !centers || !radii) return DART_E_BADARG;
    if (n == 0) return DART_OK;
    if (g->cell_bytes == 8)
        map_add_spheres_kernel<double><<<n, 256, 0, (cudaStream_t)stream>>>(*g, (double *)occ_writable, n, centers, radii, value);
    else
        map_add_spheres_kernel<float><<<n, 256, 0, (cudaStream_t)stream>>>(*g, (float *)occ_writable, n, centers, radii, (float)value);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}

int dart_map_signed_distance(const dart_grid *g, double threshold, float *phi_out, int32_t *sq_scratch,
                             void *stream)
{
    if (check_grid(g) || !sq_scratch) return DART_E_BADARG;
    return edt<float>(*g, threshold, phi_out, nullptr, 0.0, 0.0, sq_scratch, (cudaStream_t)stream);
}

int dart_map_clearance_field(const dart_grid *g, double threshold, double safety_distance, double free_level,
                             void *field_out, int32_t *sq_scratch, void *stream)
{
    if (check_grid(g) || !field_out || !sq_scratch || !(safety_distance >= 0.0) || !isfinite(safety_distance) ||
        !isfinite(free_level))
        return DART_E_BADARG;
    if (g->cell_bytes == 8)
        return edt<double>(*g, threshold, nullptr, (double *)field_out, safety_distance, free_level, sq_scratch,
                           (cudaStream_t)stream);
    return edt<float>(*g, threshold, nullptr, (float *)field_out, safety_distance, free_level, sq_scratch,
                      (cudaStream_t)stream);
}

} /* extern "C" */
