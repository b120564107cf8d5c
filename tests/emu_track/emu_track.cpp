/*
 * tests/emu_track/emu_track.cpp -- TEST INFRASTRUCTURE.
 * The kernel core (dart_planner_b200/csrc/se3mpc_core.cuh) compiled for the HOST with a one-lane
 * group in the tracking modes: gradient_mode 7 (mode 3 with a per-timestep reference) and 8 (mode 6
 * with it), so the CPU-only test tier runs the kernel's own tracking terms, rollout, adjoint,
 * line-search backups, context switch and L-BFGS-B control flow against tests/track_oracle.  Build
 * policies as in tests/emu_rollout: register-rich (latency) or register-capped (throughput) build,
 * and the two-phase schedule's context switch into a NaN-poisoned second solver, which re-reads the
 * reference by problem index as the kernel does.  The product never loads this library.
 */
#include <stdlib.h>

#include "../../dart_planner_b200/csrc/se3mpc_core.cuh"

using namespace dartb200;

static int g_ls_shared = 0; /* 1: the register-capped build's policies */
static int g_two_phase = 0; /* 1: first iteration, save the context, a NEW solver restores and finishes */
extern "C" void emt_set_policy(int ls_shared, int two_phase)
{
    g_ls_shared = ls_shared;
    g_two_phase = two_phase;
}

/* ref: the problem's [6T] column (rows 3j+c position, 3T+3j+c velocity; stride 1) */
template <int TPL, int GM, bool LSS>
static void solve_one(const dart_se3mpc_params &P, const double *p0, const double *v0, int has_goal,
                      const double *ref, int T, int start, const double *xw, double *x_out, double *acc, double *att,
                      double *rates, double *thrust, SolveStats &st, const SpherePenalty *sph)
{
    using ST = Solver<SeqGroup, TPL, GM, LSS, true>;
    double smem[SM_DOUBLES], smem2[SM_DOUBLES];
    for (int i = 0; i < SM_DOUBLES; ++i) smem[i] = smem2[i] = 0.0 / 0.0; /* NaN-poison: catches stale reads */
    static double ws[MMAX][9 * TPL], wy[MMAX][9 * TPL], ws2[MMAX][9 * TPL], wy2[MMAX][9 * TPL];
    for (int j = 0; j < MMAX; ++j)
        for (int i = 0; i < 9 * TPL; ++i) ws[j][i] = wy[j][i] = ws2[j][i] = wy2[j][i] = 0.0 / 0.0;
    ST sv(P, smem, ws, wy), sv2(P, smem2, ws2, wy2);
    const int N = P.horizon;
    if constexpr (ST::SPHERES) {
        sv.obs = *sph;
        sv2.obs = *sph;
    }
    sv.has_goal = has_goal != 0;
    for (int c = 0; c < 3; ++c) sv.goal[c] = 0.0; /* not read in these modes, as in the kernel */
    sv.set_reference(ref, 1, T, start);
    if (xw)
        sv.warm_start(p0, v0, [&](int row) { return xw[row]; });
    else
        sv.cold_start(p0, v0);
    ST *out = &sv;
    if (g_two_phase && LSS) {
        sv.begin();
        if (sv.task == 0) sv.template iterate<true>();
        if (sv.task == 0) {
            static double ctx[ST::ctx_doubles(1)];
            for (int i = 0; i < ST::ctx_doubles(1); ++i) ctx[i] = 0.0 / 0.0;
            if (sv.col > 1) abort();
            sv.save_context(ctx, 1, 1357);
            for (int k = 0; k < TPL; ++k)
                for (int c = 0; c < 3; ++c) sv2.rp[k][c] = sv2.rv[k][c] = 0.0 / 0.0;
            if (sv2.restore_context(ctx, 1) != 1357) abort();
            sv2.set_reference(ref, 1, T, start);
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
}

template <int TPL, int GM>
static void dispatch(const dart_se3mpc_params &P, const double *p0, const double *v0, int hg, const double *ref, int T,
                     int start, const double *xw, double *x, double *acc, double *att, double *rates, double *thrust,
                     SolveStats &st, const SpherePenalty *sph)
{
    if (g_ls_shared)
        solve_one<TPL, GM, true>(P, p0, v0, hg, ref, T, start, xw, x, acc, att, rates, thrust, st, sph);
    else
        solve_one<TPL, GM, false>(P, p0, v0, hg, ref, T, start, xw, x, acc, att, rates, thrust, st, sph);
}

/* ref: [B][6T] (each problem's column of the dart_track_ref block); spheres (mode 8) [n][4] */
extern "C" int emt_solve_batch(const dart_se3mpc_params *P, long B, const double *p0, const double *v0,
                               const unsigned char *has_goal, const double *x_warm, const double *ref, int T,
                               int start, const double *spheres, int n_spheres, double margin, double *x,
                               double *cost, int *nit, int *nfev, int *status, int *task, double *acc, double *att,
                               double *rates, double *thrust)
{
    const int N = P->horizon, n = 9 * N, gm = P->gradient_mode;
    if (N < 1 || N > 16 || P->max_corrections < 1 || P->max_corrections > MMAX) return -2;
    if (gm != 7 && gm != 8) return -3;
    if (T < 1 || start < 0 || !ref) return -1;
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
        const double *pb = p0 + 3 * b, *vb = v0 + 3 * b, *rb0 = ref + 6L * T * b;
        double *xb = x + (long)n * b, *ab = acc + 3L * N * b, *tb = att + 3L * N * b, *rb = rates + 3L * N * b,
               *hb = thrust + (long)N * b;
        if (N <= 8)
            (gm == 7 ? dispatch<8, 7> : dispatch<8, 8>)(*P, pb, vb, hg, rb0, T, start, xw, xb, ab, tb, rb, hb, st, &sph);
        else
            (gm == 7 ? dispatch<16, 7> : dispatch<16, 8>)(*P, pb, vb, hg, rb0, T, start, xw, xb, ab, tb, rb, hb, st,
                                                         &sph);
        cost[b] = st.f; nit[b] = st.nit; nfev[b] = st.nfev; status[b] = st.status; task[b] = st.task;
    }
    return 0;
}
