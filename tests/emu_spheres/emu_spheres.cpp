/*
 * tests/emu_spheres/emu_spheres.cpp -- TEST INFRASTRUCTURE.
 * The kernel core (dart_planner_b200/csrc/se3mpc_core.cuh) compiled for the HOST with a one-lane
 * group in the sphere-penalty modes: gradient_mode 5 (mode 0 + spheres) and 6 (mode 3 + spheres),
 * so the CPU-only test tier runs the kernel's own penalty, line-search backups, context switch and
 * L-BFGS-B control flow against tests/sphere_oracle.  Build policies as in tests/emu and
 * tests/emu_rollout: register-rich (latency) or register-capped (throughput) build, the 7-slot
 * instantiation (mode 5 only: the lateral thrust stays exactly zero), and the two-phase schedule's
 * context switch into a NaN-poisoned second solver.  The product never loads this library.
 */
#include <stdlib.h>

#include "../../dart_planner_b200/csrc/se3mpc_core.cuh"

using namespace dartb200;

static int g_ls_shared = 0;  /* 1: the register-capped build's policies */
static int g_two_phase = 0;  /* 1: first iteration, save the context, a NEW solver restores and finishes */
static int g_seven_slot = 0; /* 1 (mode 5): the TILT=false instantiation, cold and warm */
extern "C" void ems_set_policy(int ls_shared, int two_phase, int seven_slot)
{
    g_ls_shared = ls_shared;
    g_two_phase = two_phase;
    g_seven_slot = seven_slot;
}

template <int TPL, int GM, bool LSS, bool TILT>
static int solve_one(const dart_se3mpc_params &P, const double *p0, const double *v0, const double *goal, int has_goal,
                     const double *xw, double *x_out, double *acc, double *att, double *rates, double *thrust,
                     SolveStats &st, const SpherePenalty &sph)
{
    using ST = Solver<SeqGroup, TPL, GM, LSS, TILT>;
    double smem[SM_DOUBLES], smem2[SM_DOUBLES];
    for (int i = 0; i < SM_DOUBLES; ++i) smem[i] = smem2[i] = 0.0 / 0.0; /* NaN-poison: catches stale reads */
    static double ws[MMAX][9 * TPL], wy[MMAX][9 * TPL], ws2[MMAX][9 * TPL], wy2[MMAX][9 * TPL];
    for (int j = 0; j < MMAX; ++j)
        for (int i = 0; i < 9 * TPL; ++i) ws[j][i] = wy[j][i] = ws2[j][i] = wy2[j][i] = 0.0 / 0.0;
    ST sv(P, smem, ws, wy), sv2(P, smem2, ws2, wy2);
    const int N = P.horizon;
    sv.obs = sph;
    sv2.obs = sph;
    sv.has_goal = has_goal != 0;
    for (int c = 0; c < 3; ++c) sv.goal[c] = goal[c];
    if (xw) {
        sv.warm_start(p0, v0, [&](int row) { return xw[row]; });
        if (!TILT)
            for (int k = 0; k < N; ++k)
                if (sv.x[k * 9 + 6] != 0.0 || sv.x[k * 9 + 7] != 0.0) return -4; /* the 7-slot promise */
    } else
        sv.cold_start(p0, v0);
    ST *out = &sv;
    if (g_two_phase && LSS) {
        sv.begin();
        if (sv.task == 0) sv.template iterate<true>();
        if (sv.task == 0) {
            static double ctx[ST::ctx_doubles(1)];
            for (int i = 0; i < ST::ctx_doubles(1); ++i) ctx[i] = 0.0 / 0.0;
            if (sv.col > 1) abort();
            sv.save_context(ctx, 1, 2468);
            for (int c = 0; c < (int)(sizeof(sv2.gobs) / sizeof(double)); ++c) sv2.gobs[c] = 0.0 / 0.0;
            if (sv2.restore_context(ctx, 1) != 2468) abort();
            while (sv2.task == 0) sv2.template iterate<false>();
            out = &sv2;
        }
        out->finish(st);
    } else
        sv.minimize(st);
    for (int k = 0; k < N; ++k)
        for (int q = 0; q < 9; ++q) x_out[(q / 3) * 3 * N + 3 * k + q % 3] = out->x[k * 9 + q];
    out->extract([&](int k, double ax, double ay, double az, double a0, double a1, double a2, double w0, double w1,
                     double w2, double th) {
        acc[3 * k] = ax; acc[3 * k + 1] = ay; acc[3 * k + 2] = az;
        att[3 * k] = a0; att[3 * k + 1] = a1; att[3 * k + 2] = a2;
        rates[3 * k] = w0; rates[3 * k + 1] = w1; rates[3 * k + 2] = w2;
        thrust[k] = th;
    });
    return 0;
}

template <int TPL, int GM>
static int dispatch(const dart_se3mpc_params &P, const double *p0, const double *v0, const double *goal, int hg,
                    const double *xw, double *x, double *acc, double *att, double *rates, double *thrust,
                    SolveStats &st, const SpherePenalty &sph)
{
#define EMS_CALL(L, T) solve_one<TPL, GM, L, T>(P, p0, v0, goal, hg, xw, x, acc, att, rates, thrust, st, sph)
    if (GM == 5 && g_seven_slot) return g_ls_shared ? EMS_CALL(true, false) : EMS_CALL(false, false);
    return g_ls_shared ? EMS_CALL(true, true) : EMS_CALL(false, true);
#undef EMS_CALL
}

extern "C" int ems_solve_batch(const dart_se3mpc_params *P, long B, const double *p0, const double *v0,
                               const double *goal, const unsigned char *has_goal, const double *x_warm,
                               const double *spheres, int n_spheres, double margin, double *x, double *cost, int *nit,
                               int *nfev, int *status, int *task, double *acc, double *att, double *rates,
                               double *thrust)
{
    const int N = P->horizon, n = 9 * N, gm = P->gradient_mode;
    if (N < 1 || N > 32 || P->max_corrections < 1 || P->max_corrections > MMAX) return -2;
    if (gm != 5 && gm != 6) return -3;
    if (n_spheres < 0 || (n_spheres > 0 && !spheres)) return -1;
    SpherePenalty sph;
    sph.s = spheres;
    sph.n = n_spheres;
    sph.w = P->w_obstacle;
    sph.margin = margin;
    for (long b = 0; b < B; ++b) {
        SolveStats st;
        const double *xw = x_warm ? x_warm + (long)n * b : nullptr;
        const int hg = has_goal ? has_goal[b] : 1;
        const double *pb = p0 + 3 * b, *vb = v0 + 3 * b, *gb = goal + 3 * b;
        double *xb = x + (long)n * b, *ab = acc + 3L * N * b, *tb = att + 3L * N * b, *rb = rates + 3L * N * b,
               *hb = thrust + (long)N * b;
        int rc;
        if (N <= 8)
            rc = (gm == 5 ? dispatch<8, 5> : dispatch<8, 6>)(*P, pb, vb, gb, hg, xw, xb, ab, tb, rb, hb, st, sph);
        else if (N <= 20)
            rc = (gm == 5 ? dispatch<20, 5> : dispatch<20, 6>)(*P, pb, vb, gb, hg, xw, xb, ab, tb, rb, hb, st, sph);
        else
            rc = (gm == 5 ? dispatch<32, 5> : dispatch<32, 6>)(*P, pb, vb, gb, hg, xw, xb, ab, tb, rb, hb, st, sph);
        if (rc) return rc;
        cost[b] = st.f; nit[b] = st.nit; nfev[b] = st.nfev; status[b] = st.status; task[b] = st.task;
    }
    return 0;
}

/* the core's penalty alone at npos positions [npos][3]: f [npos], grad [npos][3] */
extern "C" void ems_penalty(const double *spheres, int n_spheres, double w, double margin, long npos, const double *P,
                            double *f, double *grad)
{
    SpherePenalty sph;
    sph.s = spheres;
    sph.n = n_spheres;
    sph.w = w;
    sph.margin = margin;
    for (long i = 0; i < npos; ++i) f[i] = sph.eval(P[3 * i], P[3 * i + 1], P[3 * i + 2], grad + 3 * i);
}
