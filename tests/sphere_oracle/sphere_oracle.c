/*
 * tests/sphere_oracle/sphere_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU oracle of the sphere obstacle penalty (gradient_mode 5 = mode 0 + spheres, gradient_mode 6 =
 * mode 3 + spheres; an extension -- the reference builds the constraint |P_k - c|^2 >= (r +
 * safety_margin)^2, se3_mpc_planner.py:499-514, and never passes it to minimize).  Built on the
 * reference oracle (oracle/se3mpc_oracle.c, oracle/lbfgsb_oracle.c) and the dynamics-consistent
 * oracle (tests/rollout_oracle/rollout_oracle.c), compiled into the same library:
 *   mode 5: the reference objective and gradient (orc_objective / orc_gradient) plus the penalty on
 *           the position variables, on the reference oracle's L-BFGS-B driver over the 9N variables,
 *           as orc_solve_batch_grid adds the grid penalty;
 *   mode 6: rol_fg's rollout and sequential adjoint with the penalty's gradient entering dP, over
 *           the 3N thrusts.
 * Plain sequential restatement: no lane groups, no scans.
 *
 * The penalty (the same statement as include/dart_se3mpc.h, dart_spheres, and SpherePenalty in
 * dart_planner_b200/csrc/se3mpc_core.cuh).  For spheres j = 0 .. n-1 in list order, each product and
 * sum individually rounded (this file is compiled with -ffp-contract=off):
 *   e = P - c_j,  d2 = (e_x e_x + e_y e_y) + e_z e_z,  R = r_j + margin,  h = R R - d2,
 *   h > 0:  f += w (h h),  grad += ((-4 w) h) e,
 * f starting at +0 and grad at -0 for each position.
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

double sph_penalty(const sph_list *L, const double *P, double *grad)
{
    double f = 0.0;
    grad[0] = grad[1] = grad[2] = -0.0;
    for (int j = 0; j < L->n; ++j) {
        const double *c = L->s + 4 * j;
        const double e[3] = {P[0] - c[0], P[1] - c[1], P[2] - c[2]};
        const double d2 = (e[0] * e[0] + e[1] * e[1]) + e[2] * e[2];
        const double R = c[3] + L->margin;
        const double h = R * R - d2;
        if (h > 0.0) {
            f += L->w * (h * h);
            const double k = (-4.0 * L->w) * h;
            for (int a = 0; a < 3; ++a) grad[a] += k * e[a];
        }
    }
    return f;
}

/* mode 5: f and g at the packed x [P | V | T] */
double sph_fg5(const orc_params *p, const double *goal, const sph_list *L, const double *x, double *g)
{
    orc_gradient(p, x, goal, g);
    double f = orc_objective(p, x, goal);
    for (int k = 0; k < p->horizon; ++k) {
        double gr[3];
        f += sph_penalty(L, x + 3 * k, gr);
        for (int a = 0; a < 3; ++a) g[3 * k + a] += gr[a];
    }
    return f;
}

/* mode 6: f at the rolled-out x and df/dT by the sequential adjoint (rol_fg with the sphere term);
 * x (9N) is scratch that receives the rolled-out vector */
double sph_fg6(const orc_params *p, const double *p0, const double *v0, const double *goal, const sph_list *L,
               const double *T, double *x, double *gT)
{
    const int N = p->horizon;
    const double hover = p->mass * p->gravity, dt = p->dt, hdt2 = 0.5 * (dt * dt);
    memcpy(x + 6 * N, T, sizeof(double) * 3 * N);
    rol_rollout(p, p0, v0, x);
    double f = orc_objective(p, x, goal);
    const double *P = x, *V = x + 3 * N;
    double mu[3] = {0.0, 0.0, 0.0}, nu[3] = {0.0, 0.0, 0.0}, gr[3];
    for (int k = 0; k < N; ++k) f += sph_penalty(L, P + 3 * k, gr);
    for (int k = N - 1; k >= 0; --k) {
        sph_penalty(L, P + 3 * k, gr);
        for (int c = 0; c < 3; ++c) {
            double gp = 0.0;
            if (goal) {
                const double e = P[3 * k + c] - goal[c];
                gp = 2 * p->w_pos * e;
                if (k == N - 1) gp += 2 * 10 * p->w_pos * e;
            }
            gp += gr[c];
            const double gv = 2 * p->w_vel * V[3 * k + c];
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
    const double *p0, *v0, *goal;
    const sph_list *L;
    double *x;
} fg_ctx;

static double fg5(int n, const double *x, double *g, void *user)
{
    (void)n;
    fg_ctx *c = (fg_ctx *)user;
    return sph_fg5(c->p, c->goal, c->L, x, g);
}

static double fg6(int n, const double *t, double *g, void *user)
{
    (void)n;
    fg_ctx *c = (fg_ctx *)user;
    return sph_fg6(c->p, c->p0, c->v0, c->goal, c->L, t, c->x, g);
}

/* one solve in mode 5 or 6: the start of :282-359 / :294-327, the boxes of :378-402, SciPy's
 * wrapper semantics (orc_lbfgsb), the extraction of :582-654.  x: 9N out. */
static int solve_one(const orc_params *p, int mode, const double *p0, const double *v0, const double *goal,
                     const double *x_warm, const sph_list *L, double *x, double *acc, double *att, double *rates,
                     double *thrust, orc_stats *st)
{
    const int N = p->horizon, n = 9 * N;
    double *buf = (double *)malloc(sizeof(double) * 21 * N);
    int32_t *nbd = (int32_t *)malloc(sizeof(int32_t) * n);
    if (!buf || !nbd) {
        free(buf);
        free(nbd);
        return -1;
    }
    double *lo = buf, *hi = buf + 9 * N, *t = buf + 18 * N;
    if (x_warm)
        orc_warm_start(p, p0, v0, x_warm, x);
    else
        orc_cold_start(p, p0, v0, goal, x);
    orc_bounds(p, lo, hi);
    for (int i = 0; i < n; ++i) nbd[i] = 2;
    fg_ctx c = {p, p0, v0, goal, L, x};
    const double eps = 2.220446049250313e-16;
    int rc;
    if (mode == 5) {
        rc = orc_lbfgsb(n, p->max_corrections, x, lo, hi, nbd, fg5, &c, p->ftol / eps, p->gtol, p->max_iterations,
                        p->max_fun, p->max_linesearch, st);
    } else {
        memcpy(t, x + 6 * N, sizeof(double) * 3 * N);
        rc = orc_lbfgsb(3 * N, p->max_corrections, t, lo + 6 * N, hi + 6 * N, nbd, fg6, &c, p->ftol / eps, p->gtol,
                        p->max_iterations, p->max_fun, p->max_linesearch, st);
        memcpy(x + 6 * N, t, sizeof(double) * 3 * N);
        rol_rollout(p, p0, v0, x);
    }
    orc_extract(p, x, acc, att, rates, thrust);
    free(buf);
    free(nbd);
    return rc;
}

typedef struct {
    const orc_params *p;
    int mode;
    int64_t b0, b1;
    const double *p0, *v0, *goal, *x_warm;
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
        const double *goal = (j->has_goal && !j->has_goal[b]) ? NULL : j->goal + 3 * b;
        const double *xw = j->x_warm ? j->x_warm + (int64_t)n * b : NULL;
        const int rc = solve_one(j->p, j->mode, j->p0 + 3 * b, j->v0 + 3 * b, goal, xw, j->L, j->x + (int64_t)n * b,
                                 j->acc + (int64_t)3 * N * b, j->att + (int64_t)3 * N * b,
                                 j->rates + (int64_t)3 * N * b, j->thrust + (int64_t)N * b, &st);
        if (rc) j->rc = rc;
        j->cost[b] = st.f;
        j->nit[b] = st.nit;
        j->nfev[b] = st.nfev;
        j->status[b] = st.status;
        j->task[b] = st.task;
    }
    return NULL;
}

/* B problems in mode 5 or 6, inputs [B][3]; every output is required */
int sph_solve_batch(const orc_params *p, int mode, int64_t B, const double *p0, const double *v0, const double *goal,
                    const uint8_t *has_goal, const double *x_warm, const double *spheres, int32_t n_spheres,
                    double w, double margin, double *x, double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                    int32_t *task, double *acc, double *att, double *rates, double *thrust, int nthreads)
{
    if (mode != 5 && mode != 6) return -2;
    const sph_list L = {spheres, n_spheres, w, margin};
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
        *j = (job){p, mode, B * i / nthreads, B * (i + 1) / nthreads, p0, v0, goal, x_warm, has_goal, &L,
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

/* the penalty and its gradient at npos positions [npos][3] (grad [npos][3]); returns the sum of f
 * in position order */
double sph_penalty_batch(const double *spheres, int32_t n_spheres, double w, double margin, int64_t npos,
                         const double *P, double *f_out, double *grad)
{
    const sph_list L = {spheres, n_spheres, w, margin};
    double s = 0.0;
    for (int64_t i = 0; i < npos; ++i) {
        const double f = sph_penalty(&L, P + 3 * i, grad + 3 * i);
        if (f_out) f_out[i] = f;
        s += f;
    }
    return s;
}

/* mode 5 / 6 objective and gradient at one point (mode 5: x [9N] -> g [9N]; mode 6: T [3N] -> gT
 * [3N], x_scratch [9N] receives the rollout) */
double sph_fg(const orc_params *p, int mode, const double *p0, const double *v0, const double *goal,
              const double *spheres, int32_t n_spheres, double w, double margin, const double *v, double *x_scratch,
              double *g)
{
    const sph_list L = {spheres, n_spheres, w, margin};
    if (mode == 5) return sph_fg5(p, goal, &L, v, g);
    return sph_fg6(p, p0, v0, goal, &L, v, x_scratch, g);
}
