/*
 * tests/rollout_oracle/rollout_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU oracle of the dynamics-consistent solve mode (gradient_mode 3, and 4 with the occupancy-grid
 * penalty; an extension -- the reference never passes its dynamics residual to its optimiser).
 * Built on the reference oracle (oracle/se3mpc_oracle.c, oracle/lbfgsb_oracle.c, compiled into the
 * same library): the generic L-BFGS-B driver runs over the 3N thrusts, the objective is the
 * reference objective (orc_objective, se3_mpc_planner.py:516-550) at the rolled-out vector, the
 * gradient its exact adjoint.  Plain sequential restatement: no lane groups, no scans.
 *
 * Rollout: the plant model of se3_mpc_planner.py:430-431, :445-459 from (p0, v0):
 *   a_k = T_k/m - g e3,  P_{k+1} = (P_k + V_k dt) + (0.5 a_k) dt^2,  V_{k+1} = V_k + a_k dt.
 */
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include "../../oracle/se3mpc_oracle.h"

/* fills P, V of the packed x [P | V | T] (se3_mpc_planner.py:361-376) from its T rows */
void rol_rollout(const orc_params *p, const double *p0, const double *v0, double *x)
{
    const int N = p->horizon;
    double *P = x, *V = x + 3 * N;
    const double *T = x + 6 * N;
    const double dt = p->dt, dt2 = dt * dt;
    for (int c = 0; c < 3; ++c) {
        P[c] = p0[c];
        V[c] = v0[c];
    }
    for (int k = 0; k + 1 < N; ++k)
        for (int c = 0; c < 3; ++c) {
            const double a = T[3 * k + c] / p->mass + (c == 2 ? -p->gravity : -0.0);
            P[3 * (k + 1) + c] = (P[3 * k + c] + V[3 * k + c] * dt) + (0.5 * a) * dt2;
            V[3 * (k + 1) + c] = V[3 * k + c] + a * dt;
        }
}

/* f at the rolled-out x (+ the grid penalty on the positions when grid != NULL) and df/dT by the
 * sequential adjoint:
 *   mu_{N-1} = df/dP_{N-1},  nu_{N-1} = df/dV_{N-1},
 *   mu_k = df/dP_k + mu_{k+1},  nu_k = (df/dV_k + nu_{k+1}) + dt mu_{k+1},
 *   df/dT_k = direct terms + ((0.5 dt^2) mu_{k+1} + dt nu_{k+1}) / m   for k < N-1.
 * x (9N) is scratch that receives the rolled-out vector. */
double rol_fg(const orc_params *p, const double *p0, const double *v0, const double *goal,
              const orc_grid *grid, double w_obs, double free_level, const double *T, double *x, double *gT)
{
    const int N = p->horizon;
    const double hover = p->mass * p->gravity, dt = p->dt, hdt2 = 0.5 * (dt * dt);
    memcpy(x + 6 * N, T, sizeof(double) * 3 * N);
    rol_rollout(p, p0, v0, x);
    double f = orc_objective(p, x, goal);
    const double *P = x, *V = x + 3 * N;
    double mu[3] = {0.0, 0.0, 0.0}, nu[3] = {0.0, 0.0, 0.0}, gr[3] = {0.0, 0.0, 0.0};
    if (grid)
        for (int k = 0; k < N; ++k) f += orc_grid_penalty(grid, w_obs, free_level, P + 3 * k, gr);
    for (int k = N - 1; k >= 0; --k) {
        if (grid) orc_grid_penalty(grid, w_obs, free_level, P + 3 * k, gr);
        for (int c = 0; c < 3; ++c) {
            double gp = 0.0;
            if (goal) {
                const double e = P[3 * k + c] - goal[c];
                gp = 2 * p->w_pos * e;
                if (k == N - 1) gp += 2 * 10 * p->w_pos * e;
            }
            if (grid) gp += gr[c];
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
    const orc_grid *grid;
    double w_obs, free_level;
    double *x;
} fg_ctx;

static double fg(int n, const double *t, double *g, void *user)
{
    (void)n;
    fg_ctx *c = (fg_ctx *)user;
    return rol_fg(c->p, c->p0, c->v0, c->goal, c->grid, c->w_obs, c->free_level, t, c->x, g);
}

/* one solve: the start of :282-359 / :294-327 (orc_cold_start / orc_warm_start), its thrusts as
 * the variables with their boxes (:378-402), SciPy's wrapper semantics (orc_lbfgsb), then the
 * rollout of the result and the extraction (:582-654).  x: 9N out. */
static int solve_one(const orc_params *p, const double *p0, const double *v0, const double *goal,
                     const double *x_warm, const orc_grid *grid, double w_obs, double free_level, double *x,
                     double *acc, double *att, double *rates, double *thrust, orc_stats *st)
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
        orc_cold_start(p, p0, v0, goal, x);
    orc_bounds(p, lo, hi);
    for (int i = 0; i < 3 * N; ++i) nbd[i] = 2;
    memcpy(t, x + 6 * N, sizeof(double) * 3 * N);
    fg_ctx c = {p, p0, v0, goal, grid, w_obs, free_level, x};
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
    const double *p0, *v0, *goal, *x_warm;
    const uint8_t *has_goal;
    const orc_grid *grid;
    double w_obs, free_level;
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
        const int rc = solve_one(j->p, j->p0 + 3 * b, j->v0 + 3 * b, goal, xw, j->grid, j->w_obs, j->free_level,
                                 j->x + (int64_t)n * b, j->acc + (int64_t)3 * N * b, j->att + (int64_t)3 * N * b,
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

/* B problems, inputs [B][3]; every output is required ([B][9N], [B], [B][N][3], [B][N]) */
int rol_solve_batch(const orc_params *p, int64_t B, const double *p0, const double *v0, const double *goal,
                    const uint8_t *has_goal, const double *x_warm, double *x, double *cost, int32_t *nit,
                    int32_t *nfev, int32_t *status, int32_t *task, double *acc, double *att, double *rates,
                    double *thrust, int nthreads, const orc_grid *grid, double w_obs, double free_level)
{
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
        *j = (job){p, B * i / nthreads, B * (i + 1) / nthreads, p0, v0, goal, x_warm, has_goal, grid, w_obs,
                   free_level, x, cost, acc, att, rates, thrust, nit, nfev, status, task, 0};
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
