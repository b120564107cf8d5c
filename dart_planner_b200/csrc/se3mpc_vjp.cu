/*
 * se3mpc_vjp.cu -- C ABI of the differentiable solve (dart_se3mpc_solve_vjp_batch): the
 * vector-Jacobian product of a returned plan in gradient modes 3, 6, 7 and 8.  The device routine is
 * PlanVjp in se3mpc_core.cuh; here are the argument checks, the kernel and its launch.  One problem
 * per sub-warp of 4, 8 or 16 lanes (one timestep per lane), as the solve at these horizons; goal and
 * reference, with and without spheres, share one kernel per lane width.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "se3mpc_kernel.cuh"

extern "C" void dart_count_launch_(void);

namespace dartb200 {

template <int LANES>
__global__ void __launch_bounds__(128)
se3mpc_vjp_kernel(const __grid_constant__ dart_se3mpc_params P, const __grid_constant__ VjpArgs A)
{
    using GMap = GroupMap<LANES, 128>;
    constexpr int GPB = GMap::GPB;
    const long long rounds = (A.B + GPB - 1) / GPB;
    for (long long blk = blockIdx.x; blk < rounds; blk += gridDim.x) {
        const long long b = blk * GPB + GMap::gib();
        if (b < A.B) {
            PlanVjp<typename GroupOf<LANES>::type, 1> vjp(P);
            vjp.run(A, b);
        }
    }
}

} /* namespace dartb200 */

using namespace dartb200;

extern "C" int dart_se3mpc_solve_vjp_batch(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                           const double *p0, const double *v0, const double *goal,
                                           const uint8_t *has_goal, const double *x, const dart_track_ref *ref,
                                           const dart_spheres *spheres, const double *gx, const double *gcost,
                                           double *gp0, double *gv0, double *ggoal, double *gref, double *gw,
                                           int32_t *status, void *cuda_stream)
{
    if (!params || params->struct_size != (int)sizeof(dart_se3mpc_params)) return DART_E_BADARG;
    const int N = params->horizon;
    /* the dynamics-consistent modes without the grid penalty: 3, 6, 7 and 8 */
    const ModeInfo *m = mode_info(params->gradient_mode);
    if (!m || !m->rollout || m->grid_pen) return DART_E_BADARG;
    const bool track = m->track, sph = m->spheres;
    if (sph != (spheres != nullptr) || track != (ref != nullptr)) return DART_E_BADARG;
    if (spheres && (spheres->n < 0 || (spheres->n > 0 && !spheres->cxyzr))) return DART_E_BADARG;
    if (ref && (!ref->rows || ref->len != N || ref->start != 0)) return DART_E_BADARG;
    if (!x || !status || !p0 || !v0 || (!track && !goal) || B < 0 || ld < B) return DART_E_BADARG;
    if (N < 1) return DART_E_BADARG;
    if (N > m->max_horizon) return DART_E_UNSUPPORTED;
    if (!(params->dt > 0.0) || !(params->mass > 0.0)) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    VjpArgs a;
    a.B = B;
    a.ld = ld;
    a.p0 = p0;
    a.v0 = v0;
    a.goal = track ? nullptr : goal;
    a.has_goal = has_goal;
    a.x = x;
    a.ref = track ? ref->rows : nullptr;
    a.spheres = sph ? spheres->cxyzr : nullptr;
    a.n_spheres = sph ? spheres->n : 0;
    a.sphere_margin = sph ? spheres->margin : 0.0;
    a.gx = gx;
    a.gcost = gcost;
    a.gp0 = gp0;
    a.gv0 = gv0;
    a.ggoal = ggoal;
    a.gref = gref;
    a.gw = gw;
    a.status = status;
    const int lanes = N <= 4 ? 4 : (N <= 8 ? 8 : 16);
    const long long gpb = 128 / lanes;
    const long long blocks = (B + gpb - 1) / gpb;
    const unsigned grid = (unsigned)(blocks < (1ll << 30) ? blocks : (1ll << 30));
    cudaStream_t s = (cudaStream_t)cuda_stream;
    if (lanes == 4)
        se3mpc_vjp_kernel<4><<<grid, 128, 0, s>>>(*params, a);
    else if (lanes == 8)
        se3mpc_vjp_kernel<8><<<grid, 128, 0, s>>>(*params, a);
    else
        se3mpc_vjp_kernel<16><<<grid, 128, 0, s>>>(*params, a);
    if (cudaGetLastError() != cudaSuccess) return DART_E_CUDA;
    dart_count_launch_();
    return DART_OK;
}
