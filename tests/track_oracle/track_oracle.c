/*
 * tests/track_oracle/track_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU oracle of reference tracking (gradient_mode 7 = mode 3 with a per-timestep reference,
 * gradient_mode 8 = mode 6 with it; an extension).  Built on the reference oracle's L-BFGS-B driver
 * (oracle/lbfgsb_oracle.c) over the n = 3N thrusts, the dynamics-consistent oracle's rollout
 * (tests/rollout_oracle/rollout_oracle.c) and the sphere oracle's penalty
 * (tests/sphere_oracle/sphere_oracle.c), compiled into the same library.  Plain sequential
 * restatement: no lane groups, no scans; the sphere sum in list order.
 *
 * The definition (the same statement as include/dart_se3mpc.h, dart_track_ref, and eval_rollout in
 * dart_planner_b200/csrc/se3mpc_core.cuh; this file is compiled with -ffp-contract=off):
 *
 * Reference tracking (gradient_mode 7 = mode 3, 8 = mode 6, with a per-timestep reference).
 * For timestep k = 0..N-1, r_k is the reference position and u_k the reference velocity, sample
 * j = min(s + k, T - 1) of the reference.  Each operation is rounded on its own (no contraction):
 *   e = P_k - r_k,  ev = V_k - u_k  (per component),
 *   f += wpf_k (e.e) + w_vel (ev.ev) + w_acc |a_k|^2 + w_thrust |T_k - m g e3|^2,
 *        wpf_k = w_pos, and 11 w_pos at k = N-1,
 *   dP_k = 2 w_pos e, plus 20 w_pos e at k = N-1,   dV_k = 2 w_vel ev,
 *   mode 8 adds the sphere penalty on P_k exactly as mode 6 does.
 * has_goal = 0 turns the position terms off; the goal input is not read.  With r_k = goal and
 * u_k = +0, e and ev are the doubles of mode 3 (v - (+0) = v, -0 - (+0) = -0), so the objective
 * and gradient are mode 3's bits, and mode 8's are mode 6's.
 *
 * Here the objective is summed in orc_objective's order (every position term, every velocity term,
 * every acceleration term, every thrust term, then the terminal 10 w_pos term), so with r_k = goal
 * and u_k = +0 it is orc_objective's value bit for bit.  The reference of one problem is given as
 * P [T][3] and V [T][3].
 */
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include "../../oracle/se3mpc_oracle.h"

void rol_rollout(const orc_params *p, const double *p0, const double *v0, double *x);

typedef struct {
    const double *s; /* [n][4] cx cy cz r */
    int32_t n;
    double w, margin;
} sph_list;
double sph_penalty(const sph_list *L, const double *P, double *grad);

typedef struct {
    const double *P, *V; /* [T][3] each */
    int32_t T, start;
} trk_ref;

static inline double sum3sq(double a, double b, double c) { return (a * a + b * b) + c * c; }
static inline int64_t trk_j(const trk_ref *r, int k)
{
    const int64_t j = (int64_t)r->start + k;
    return j < r->T ? j : r->T - 1;
}

/* f at the rolled-out x and df/dT by the sequential adjoint; x (9N) is scratch that receives the
 * rolled-out vector; L == NULL: mode 7 */
double trk_fg(const orc_params *p, const double *p0, const double *v0, int pos_on, const trk_ref *r,
              const sph_list *L, const double *T, double *x, double *gT)
{
    const int N = p->horizon;
    const double hover = p->mass * p->gravity, dt = p->dt, hdt2 = 0.5 * (dt * dt);
    memcpy(x + 6 * N, T, sizeof(double) * 3 * N);
    rol_rollout(p, p0, v0, x);
    const double *P = x, *V = x + 3 * N;
    double f = 0.0;
    if (pos_on)
        for (int k = 0; k < N; ++k) {
            const double *rk = r->P + 3 * trk_j(r, k);
            f += p->w_pos * sum3sq(P[3 * k] - rk[0], P[3 * k + 1] - rk[1], P[3 * k + 2] - rk[2]);
        }
    for (int k = 0; k < N; ++k) {
        const double *uk = r->V + 3 * trk_j(r, k);
        f += p->w_vel * sum3sq(V[3 * k] - uk[0], V[3 * k + 1] - uk[1], V[3 * k + 2] - uk[2]);
    }
    for (int k = 0; k < N; ++k)
        f += p->w_acc * sum3sq(T[3 * k] / p->mass - 0.0, T[3 * k + 1] / p->mass - 0.0,
                               T[3 * k + 2] / p->mass - p->gravity);
    for (int k = 0; k < N; ++k) f += p->w_thrust * sum3sq(T[3 * k] - 0.0, T[3 * k + 1] - 0.0, T[3 * k + 2] - hover);
    if (pos_on) {
        const int k = N - 1;
        const double *rk = r->P + 3 * trk_j(r, k);
        f += 10 * p->w_pos * sum3sq(P[3 * k] - rk[0], P[3 * k + 1] - rk[1], P[3 * k + 2] - rk[2]);
    }
    double mu[3] = {0.0, 0.0, 0.0}, nu[3] = {0.0, 0.0, 0.0}, gr[3] = {-0.0, -0.0, -0.0};
    if (L)
        for (int k = 0; k < N; ++k) f += sph_penalty(L, P + 3 * k, gr);
    for (int k = N - 1; k >= 0; --k) {
        if (L) sph_penalty(L, P + 3 * k, gr);
        const double *rk = r->P + 3 * trk_j(r, k), *uk = r->V + 3 * trk_j(r, k);
        for (int c = 0; c < 3; ++c) {
            double gp = 0.0;
            if (pos_on) {
                const double e = P[3 * k + c] - rk[c];
                gp = 2 * p->w_pos * e;
                if (k == N - 1) gp += 2 * 10 * p->w_pos * e;
            }
            if (L) gp += gr[c];
            const double gv = 2 * p->w_vel * (V[3 * k + c] - uk[c]);
            const double t = T[3 * k + c];
            const double acc = t / p->mass - (c == 2 ? p->gravity : 0.0);
            double g = 2 * p->w_acc * acc / p->mass + 2 * p->w_thrust * (t - (c == 2 ? hover : 0.0));
            if (k < N - 1) g += (hdt2 * mu[c] + dt * nu[c]) / p->mass;
            gT[3 * k + c] = g;
            nu[c] = (gv + nu[c]) + dt * mu[c];
            mu[c] = gp + mu[c];
        }
    }
    return f;
}

typedef struct {
    const orc_params *p;
    const double *p0, *v0;
    int pos_on;
    const trk_ref *r;
    const sph_list *L;
    double *x;
} fg_ctx;

static double fg(int n, const double *t, double *g, void *user)
{
    (void)n;
    fg_ctx *c = (fg_ctx *)user;
    return trk_fg(c->p, c->p0, c->v0, c->pos_on, c->r, c->L, t, c->x, g);
}

/* one solve: the start of :282-359 / :294-327 (only its thrusts are kept), the thrust boxes of
 * :378-402, SciPy's wrapper semantics (orc_lbfgsb), the rollout of the result, the extraction */
static int solve_one(const orc_params *p, const double *p0, const double *v0, int pos_on, const trk_ref *r,
                     const double *x_warm, const sph_list *L, double *x, double *acc, double *att, double *rates,
                     double *thrust, orc_stats *st)
{
    const int N = p->horizon;
    double *buf = (double *)malloc(sizeof(double) * 21 * N);
    int32_t *nbd = (int32_t *)malloc(sizeof(int32_t) * 3 * N);
    if (!buf || !nbd) {
        free(buf);
        free(nbd);
        return -1;
    }
    double *lo = buf, *hi = buf + 9 * N, *t = buf + 18 * N;
    if (x_warm)
        orc_warm_start(p, p0, v0, x_warm, x);
    else
        orc_cold_start(p, p0, v0, NULL, x);
    orc_bounds(p, lo, hi);
    for (int i = 0; i < 3 * N; ++i) nbd[i] = 2;
    memcpy(t, x + 6 * N, sizeof(double) * 3 * N);
    fg_ctx c = {p, p0, v0, pos_on, r, L, x};
    const double eps = 2.220446049250313e-16;
    const int rc = orc_lbfgsb(3 * N, p->max_corrections, t, lo + 6 * N, hi + 6 * N, nbd, fg, &c, p->ftol / eps,
                              p->gtol, p->max_iterations, p->max_fun, p->max_linesearch, st);
    memcpy(x + 6 * N, t, sizeof(double) * 3 * N);
    rol_rollout(p, p0, v0, x);
    orc_extract(p, x, acc, att, rates, thrust);
    free(buf);
    free(nbd);
    return rc;
}

typedef struct {
    const orc_params *p;
    int64_t b0, b1;
    const double *p0, *v0, *ref_p, *ref_v, *x_warm;
    int32_t T, start;
    const uint8_t *has_goal;
    const sph_list *L;
    double *x, *cost, *acc, *att, *rates, *thrust;
    int32_t *nit, *nfev, *status, *task;
    int rc;
} job;

static void *worker(void *arg)
{
    job *j = (job *)arg;
    const int N = j->p->horizon, n = 9 * N;
    for (int64_t b = j->b0; b < j->b1; ++b) {
        orc_stats st;
        const trk_ref r = {j->ref_p + (int64_t)3 * j->T * b, j->ref_v + (int64_t)3 * j->T * b, j->T, j->start};
        const double *xw = j->x_warm ? j->x_warm + (int64_t)n * b : NULL;
        const int rc = solve_one(j->p, j->p0 + 3 * b, j->v0 + 3 * b, !(j->has_goal && !j->has_goal[b]), &r, xw,
                                 j->L, j->x + (int64_t)n * b, j->acc + (int64_t)3 * N * b,
                                 j->att + (int64_t)3 * N * b, j->rates + (int64_t)3 * N * b,
                                 j->thrust + (int64_t)N * b, &st);
        if (rc) j->rc = rc;
        j->cost[b] = st.f;
        j->nit[b] = st.nit;
        j->nfev[b] = st.nfev;
        j->status[b] = st.status;
        j->task[b] = st.task;
    }
    return NULL;
}

/* B problems in mode 7 (n_spheres < 0: no list) or 8; inputs [B][3], reference [B][T][3] twice;
 * every output is required */
int trk_solve_batch(const orc_params *p, int mode, int64_t B, const double *p0, const double *v0,
                    const uint8_t *has_goal, const double *x_warm, const double *ref_p, const double *ref_v,
                    int32_t T, int32_t start, const double *spheres, int32_t n_spheres, double w, double margin,
                    double *x, double *cost, int32_t *nit, int32_t *nfev, int32_t *status, int32_t *task,
                    double *acc, double *att, double *rates, double *thrust, int nthreads)
{
    if (mode != 7 && mode != 8) return -2;
    if (T < 1 || start < 0) return -3;
    const sph_list Ls = {spheres, n_spheres, w, margin};
    const sph_list *L = mode == 8 ? &Ls : NULL;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    if ((int64_t)nthreads > B) nthreads = B > 0 ? (int)B : 1;
    job *jobs = (job *)calloc(nthreads, sizeof(job));
    pthread_t *th = (pthread_t *)calloc(nthreads, sizeof(pthread_t));
    int *started = (int *)calloc(nthreads, sizeof(int));
    if (!jobs || !th || !started) {
        free(jobs);
        free(th);
        free(started);
        return -1;
    }
    for (int i = 0; i < nthreads; ++i) {
        job *j = &jobs[i];
        *j = (job){p, B * i / nthreads, B * (i + 1) / nthreads, p0, v0, ref_p, ref_v, x_warm, T, start, has_goal, L,
                   x, cost, acc, att, rates, thrust, nit, nfev, status, task, 0};
        started[i] = nthreads > 1 && pthread_create(&th[i], NULL, worker, j) == 0;
        if (!started[i]) worker(j);
    }
    int rc = 0;
    for (int i = 0; i < nthreads; ++i) {
        if (started[i]) pthread_join(th[i], NULL);
        if (jobs[i].rc) rc = jobs[i].rc;
    }
    free(jobs);
    free(th);
    free(started);
    return rc;
}

/* mode 7 / 8 objective and df/dT at thrusts T [3N] of one problem (x_scratch [9N] receives the rollout) */
double trk_fg_one(const orc_params *p, int mode, const double *p0, const double *v0, int pos_on, const double *ref_p,
                  const double *ref_v, int32_t T, int32_t start, const double *spheres, int32_t n_spheres, double w,
                  double margin, const double *thr, double *x_scratch, double *g)
{
    const trk_ref r = {ref_p, ref_v, T, start};
    const sph_list L = {spheres, n_spheres, w, margin};
    return trk_fg(p, p0, v0, pos_on, &r, mode == 8 ? &L : NULL, thr, x_scratch, g);
}
