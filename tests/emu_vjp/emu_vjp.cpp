/*
 * tests/emu_vjp/emu_vjp.cpp -- TEST INFRASTRUCTURE.
 * The device routine of the differentiable solve (PlanVjp, dart_planner_b200/csrc/se3mpc_core.cuh)
 * compiled for the HOST with a one-lane group, so the CPU-only test tier runs the kernel's own
 * tangent rollout, adjoint, sphere Hessian and conjugate gradients against tests/vjp_oracle.py.  The
 * arguments are those of dart_se3mpc_solve_vjp_batch, in host memory.  The product never loads this
 * library.
 */
#include "../../dart_planner_b200/csrc/se3mpc_core.cuh"

using namespace dartb200;

extern "C" int emv_vjp_batch(const dart_se3mpc_params *P, long B, long ld, const double *p0, const double *v0,
                             const double *goal, const unsigned char *has_goal, const double *x, const double *ref,
                             const double *spheres, int n_spheres, double margin, const double *gx,
                             const double *gcost, double *gp0, double *gv0, double *ggoal, double *gref, double *gw,
                             int *status)
{
    const int N = P->horizon, gm = P->gradient_mode;
    if (N < 1 || N > 16) return -2;
    if (gm != 3 && gm != 6 && gm != 7 && gm != 8) return -3;
    VjpArgs a;
    a.B = B;
    a.ld = ld;
    a.p0 = p0;
    a.v0 = v0;
    a.goal = goal;
    a.has_goal = has_goal;
    a.x = x;
    a.ref = ref;
    a.spheres = spheres;
    a.n_spheres = n_spheres;
    a.sphere_margin = margin;
    a.gx = gx;
    a.gcost = gcost;
    a.gp0 = gp0;
    a.gv0 = gv0;
    a.ggoal = ggoal;
    a.gref = gref;
    a.gw = gw;
    a.status = status;
    for (long b = 0; b < B; ++b) {
        PlanVjp<SeqGroup, 16> v(*P);
        v.run(a, b);
    }
    return 0;
}
