/*
 * oracle/se3mpc_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Scalar fp64 restatement of the reference planner's solve path
 * (`/root/reference/src/dart_planner/planning/se3_mpc_planner.py`) and of the mapper
 * queries next to it (`perception/explicit_geometric_mapper.py`).  Every function cites
 * the reference lines it follows.  The optimiser itself is in lbfgsb_oracle.c.
 */
#include "se3mpc_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

double orc_flops_get(void);
void orc_flops_reset(void);

/* se3_mpc_planner.py:329-359 (_create_straight_line_initialization) */
void orc_cold_start(const orc_params *p, const double *p0, const double *v0, const double *goal,
                    double *x0)
{
    const int N = p->horizon;
    double *P = x0, *V = x0 + 3 * N, *T = x0 + 6 * N;
    const double hover = p->mass * p->gravity; /* :151 */
    memset(x0, 0, sizeof(double) * 9 * N);
    for (int c = 0; c < 3; ++c) {
        P[c] = p0[c];
        V[c] = v0[c];
    }
    if (goal) {
        int den = N - 1 > 1 ? N - 1 : 1;
        for (int i = 0; i < N; ++i) {
            double alpha = (double)i / (double)den;
            for (int c = 0; c < 3; ++c) P[3 * i + c] = (1.0 - alpha) * p0[c] + alpha * goal[c];
            if (i > 0)
                for (int c = 0; c < 3; ++c)
                    V[3 * i + c] = (P[3 * i + c] - P[3 * (i - 1) + c]) / p->dt;
            T[3 * i + 2] = hover;
        }
    } else {
        for (int i = 0; i < N; ++i) {
            for (int c = 0; c < 3; ++c) P[3 * i + c] = p0[c];
            T[3 * i + 2] = hover;
        }
    }
}

/* se3_mpc_planner.py:294-327 (_create_warm_start) for a previous solution of the same
 * horizon: shift_len = N-1, so the "extend to goal" loop (:317-325) is empty. */
void orc_warm_start(const orc_params *p, const double *p0, const double *v0,
                    const double *prev_x, double *x0)
{
    const int N = p->horizon;
    double *P = x0, *V = x0 + 3 * N, *T = x0 + 6 * N;
    const double *pP = prev_x, *pV = prev_x + 3 * N, *pT = prev_x + 6 * N;
    memset(x0, 0, sizeof(double) * 9 * N);
    for (int c = 0; c < 3; ++c) {
        P[c] = p0[c];
        V[c] = v0[c];
    }
    if (N > 1) {
        for (int i = 1; i < N; ++i)
            for (int c = 0; c < 3; ++c) {
                P[3 * i + c] = pP[3 * i + c];
                V[3 * i + c] = pV[3 * i + c];
            }
        for (int i = 0; i < N - 1; ++i)
            for (int c = 0; c < 3; ++c) T[3 * i + c] = pT[3 * (i + 1) + c];
    }
}

/* se3_mpc_planner.py:378-402 (_setup_optimization_bounds) */
void orc_bounds(const orc_params *p, double *lo, double *hi)
{
    const int N = p->horizon;
    for (int i = 0; i < 3 * N; ++i) {
        lo[i] = -p->pos_bound;
        hi[i] = p->pos_bound;
        lo[3 * N + i] = -p->max_velocity;
        hi[3 * N + i] = p->max_velocity;
    }
    for (int k = 0; k < N; ++k) {
        lo[6 * N + 3 * k + 0] = -p->tilt_thrust;
        hi[6 * N + 3 * k + 0] = p->tilt_thrust;
        lo[6 * N + 3 * k + 1] = -p->tilt_thrust;
        hi[6 * N + 3 * k + 1] = p->tilt_thrust;
        lo[6 * N + 3 * k + 2] = p->min_thrust;
        hi[6 * N + 3 * k + 2] = p->max_thrust;
    }
}

static inline double sum3sq(double a, double b, double c) { return (a * a + b * b) + c * c; }

/* se3_mpc_planner.py:516-550 (_objective_function), same accumulation order */
double orc_objective(const orc_params *p, const double *x, const double *goal)
{
    const int N = p->horizon;
    const double *P = x, *V = x + 3 * N, *T = x + 6 * N;
    const double hover = p->mass * p->gravity;
    double cost = 0.0;
    if (goal)
        for (int k = 0; k < N; ++k)
            cost += p->w_pos * sum3sq(P[3 * k] - goal[0], P[3 * k + 1] - goal[1],
                                      P[3 * k + 2] - goal[2]);
    for (int k = 0; k < N; ++k) cost += p->w_vel * sum3sq(V[3 * k], V[3 * k + 1], V[3 * k + 2]);
    for (int k = 0; k < N; ++k)
        cost += p->w_acc * sum3sq(T[3 * k] / p->mass - 0.0, T[3 * k + 1] / p->mass - 0.0,
                                  T[3 * k + 2] / p->mass - p->gravity);
    for (int k = 0; k < N; ++k)
        cost += p->w_thrust * sum3sq(T[3 * k] - 0.0, T[3 * k + 1] - 0.0, T[3 * k + 2] - hover);
    if (goal) {
        const int k = N - 1;
        cost += 10 * p->w_pos *
                sum3sq(P[3 * k] - goal[0], P[3 * k + 1] - goal[1], P[3 * k + 2] - goal[2]);
    }
    return cost;
}

/* se3_mpc_planner.py:552-580 (_objective_gradient): omits the acceleration and terminal
 * terms and uses 2*w_T*T (not T - hover).  consistent_gradient=1 gives the true gradient
 * of orc_objective (extension; not the reference). */
void orc_gradient(const orc_params *p, const double *x, const double *goal, double *g)
{
    const int N = p->horizon;
    const double *P = x, *V = x + 3 * N, *T = x + 6 * N;
    const double hover = p->mass * p->gravity;
    for (int i = 0; i < 3 * N; ++i) {
        g[i] = goal ? 2 * p->w_pos * (P[i] - goal[i % 3]) : 0.0;
        g[3 * N + i] = 2 * p->w_vel * V[i];
        g[6 * N + i] = 2 * p->w_thrust * T[i];
    }
    if (p->consistent_gradient) {
        for (int k = 0; k < N; ++k)
            for (int c = 0; c < 3; ++c) {
                double t = T[3 * k + c];
                double acc = t / p->mass - (c == 2 ? p->gravity : 0.0);
                g[6 * N + 3 * k + c] =
                    2 * p->w_acc * acc / p->mass + 2 * p->w_thrust * (t - (c == 2 ? hover : 0.0));
            }
        if (goal)
            for (int c = 0; c < 3; ++c)
                g[3 * (N - 1) + c] += 2 * 10 * p->w_pos * (P[3 * (N - 1) + c] - goal[c]);
    }
}

/* se3_mpc_planner.py:582-654 (_extract_solution_from_result, _compute_attitudes_and_rates) */
void orc_extract(const orc_params *p, const double *x, double *acc, double *att, double *rates,
                 double *thrust)
{
    const int N = p->horizon;
    const double *T = x + 6 * N;
    double prevR[9];
    int have_prev = 0;
    for (int i = 0; i < N; ++i) {
        const double tx = T[3 * i], ty = T[3 * i + 1], tz = T[3 * i + 2];
        if (acc) {
            acc[3 * i] = tx / p->mass - 0.0;
            acc[3 * i + 1] = ty / p->mass - 0.0;
            acc[3 * i + 2] = tz / p->mass - p->gravity;
        }
        double mag = sqrt(tx * tx + ty * ty + tz * tz);
        if (thrust) thrust[i] = mag;
        double a[3] = {0, 0, 0}, w[3] = {0, 0, 0};
        if (mag > 1e-6) {
            double b3[3] = {tx / mag, ty / mag, tz / mag};
            /* yaw_vector = (cos 0, sin 0, 0) = (1,0,0); b1 = yaw x b3 */
            double yv[3] = {1.0, 0.0, 0.0};
            double b1[3] = {yv[1] * b3[2] - yv[2] * b3[1], yv[2] * b3[0] - yv[0] * b3[2],
                            yv[0] * b3[1] - yv[1] * b3[0]};
            double n1 = sqrt(b1[0] * b1[0] + b1[1] * b1[1] + b1[2] * b1[2]);
            if (n1 > 1e-6) {
                b1[0] /= n1;
                b1[1] /= n1;
                b1[2] /= n1;
            } else {
                b1[0] = 1;
                b1[1] = 0;
                b1[2] = 0;
            }
            double b2[3] = {b3[1] * b1[2] - b3[2] * b1[1], b3[2] * b1[0] - b3[0] * b1[2],
                            b3[0] * b1[1] - b3[1] * b1[0]};
            double R[9] = {b1[0], b2[0], b3[0], b1[1], b2[1], b3[1], b1[2], b2[2], b3[2]};
            a[0] = atan2(R[7], R[8]);
            a[1] = asin(-R[6]);
            a[2] = atan2(R[3], R[0]);
            if (have_prev) {
                double Rd[9], M[9];
                for (int k = 0; k < 9; ++k) Rd[k] = (R[k] - prevR[k]) / p->dt;
                for (int r = 0; r < 3; ++r)
                    for (int c = 0; c < 3; ++c)
                        M[3 * r + c] = R[0 * 3 + r] * Rd[0 * 3 + c] + R[1 * 3 + r] * Rd[1 * 3 + c] +
                                       R[2 * 3 + r] * Rd[2 * 3 + c];
                w[0] = M[7];
                w[1] = M[2];
                w[2] = M[3];
            }
            memcpy(prevR, R, sizeof(R));
            have_prev = 1;
        }
        if (att) memcpy(att + 3 * i, a, sizeof(a));
        if (rates) memcpy(rates + 3 * i, w, sizeof(w));
    }
}

typedef struct {
    const orc_params *p;
    const double *goal;
    const orc_grid *grid; /* NULL: no obstacle penalty */
    double w_obs, free_level;
} fg_ctx;

static double grid_cell(const orc_grid *g, int kx, int ky, int kz)
{
    const int ix = kx - g->ox, iy = ky - g->oy, iz = kz - g->oz;
    if (ix < 0 || iy < 0 || iz < 0 || ix >= g->nx || iy >= g->ny || iz >= g->nz) return g->prior;
    const int64_t i = ((int64_t)iz * g->ny + iy) * g->nx + ix;
    return g->occ64 ? g->occ64[i] : (double)g->occ[i];
}

/* Occupancy-grid obstacle penalty (EXTENSION -- the reference solve has no obstacle term, SURVEY
 * 0.3; parity unpinned, this is the definition both the kernel and this oracle follow):
 *   o(p)  = trilinear interpolation of the occupancy over voxel CENTRES ((k+0.5)*res)
 *   rho   = max(0, o(p) - free_level)
 *   f_obs = w * rho^2,   grad = 2 w rho * grad o(p)
 * summed over the N positions of the horizon. */
double orc_grid_penalty(const orc_grid *g, double w, double free_level, const double *p, double *grad)
{
    double u[3], t[3];
    int i[3];
    for (int c = 0; c < 3; ++c) {
        u[c] = p[c] / g->resolution - 0.5;
        const double fl = floor(u[c]);
        i[c] = (int)fl;
        t[c] = u[c] - fl;
    }
    const double c000 = grid_cell(g, i[0], i[1], i[2]), c100 = grid_cell(g, i[0] + 1, i[1], i[2]);
    const double c010 = grid_cell(g, i[0], i[1] + 1, i[2]), c110 = grid_cell(g, i[0] + 1, i[1] + 1, i[2]);
    const double c001 = grid_cell(g, i[0], i[1], i[2] + 1), c101 = grid_cell(g, i[0] + 1, i[1], i[2] + 1);
    const double c011 = grid_cell(g, i[0], i[1] + 1, i[2] + 1), c111 = grid_cell(g, i[0] + 1, i[1] + 1, i[2] + 1);
    const double sx = 1.0 - t[0], sy = 1.0 - t[1], sz = 1.0 - t[2];
    const double c00 = c000 * sx + c100 * t[0], c10 = c010 * sx + c110 * t[0];
    const double c01 = c001 * sx + c101 * t[0], c11 = c011 * sx + c111 * t[0];
    const double c0 = c00 * sy + c10 * t[1], c1 = c01 * sy + c11 * t[1];
    const double o = c0 * sz + c1 * t[2];
    const double rho = o - free_level;
    grad[0] = grad[1] = grad[2] = 0.0;
    if (!(rho > 0.0)) return 0.0;
    const double d00 = c100 - c000, d10 = c110 - c010, d01 = c101 - c001, d11 = c111 - c011;
    const double gx = ((d00 * sy + d10 * t[1]) * sz + (d01 * sy + d11 * t[1]) * t[2]) / g->resolution;
    const double gy = ((c10 - c00) * sz + (c11 - c01) * t[2]) / g->resolution;
    const double gz = (c1 - c0) / g->resolution;
    const double k = 2.0 * w * rho;
    grad[0] = k * gx;
    grad[1] = k * gy;
    grad[2] = k * gz;
    return w * (rho * rho);
}

static double planner_fg(int n, const double *x, double *g, void *user)
{
    (void)n;
    fg_ctx *c = (fg_ctx *)user;
    orc_gradient(c->p, x, c->goal, g);
    double f = orc_objective(c->p, x, c->goal);
    if (c->grid) {
        const int N = c->p->horizon;
        for (int k = 0; k < N; ++k) {
            double gr[3];
            f += orc_grid_penalty(c->grid, c->w_obs, c->free_level, x + 3 * k, gr);
            for (int a = 0; a < 3; ++a) g[3 * k + a] += gr[a];
        }
    }
    return f;
}

/* se3_mpc_planner.py:230-280 (_solve_se3_mpc) */
static int solve_impl(const orc_params *p, const double *p0, const double *v0, const double *goal,
                      const double *x_warm, double *x, double *acc, double *att, double *rates,
                      double *thrust, orc_stats *st, const orc_grid *grid, double w_obs,
                      double free_level);

int orc_solve(const orc_params *p, const double *p0, const double *v0, const double *goal,
              const double *x_warm, double *x, double *acc, double *att, double *rates,
              double *thrust, orc_stats *st)
{
    return solve_impl(p, p0, v0, goal, x_warm, x, acc, att, rates, thrust, st, NULL, 0.0, 0.0);
}

static int solve_impl(const orc_params *p, const double *p0, const double *v0, const double *goal,
                      const double *x_warm, double *x, double *acc, double *att, double *rates,
                      double *thrust, orc_stats *st, const orc_grid *grid, double w_obs,
                      double free_level)
{
    const int N = p->horizon, n = 9 * N;
    double *lo = (double *)malloc(sizeof(double) * 2 * n);
    int32_t *nbd = (int32_t *)malloc(sizeof(int32_t) * n);
    if (!lo || !nbd) {
        free(lo);
        free(nbd);
        return -1;
    }
    double *hi = lo + n;
    if (x_warm)
        orc_warm_start(p, p0, v0, x_warm, x);
    else
        orc_cold_start(p, p0, v0, goal, x);
    orc_bounds(p, lo, hi);
    for (int i = 0; i < n; ++i) nbd[i] = 2;
    fg_ctx ctx = {p, goal, grid, w_obs, free_level};
    const double eps = 2.220446049250313e-16;
    /* per-evaluation cost of the reference objective + gradient (SURVEY 8d: 48N+10, 12N) */
    int rc = orc_lbfgsb(n, p->max_corrections, x, lo, hi, nbd, planner_fg, &ctx, p->ftol / eps,
                        p->gtol, p->max_iterations, p->max_fun, p->max_linesearch, st);
    if (st) st->flops += (double)st->nfev * (60.0 * N + 10.0) + 90.0 * N;
    orc_extract(p, x, acc, att, rates, thrust);
    free(lo);
    free(nbd);
    return rc;
}

typedef struct {
    const orc_params *p;
    int64_t b0, b1;
    const double *p0, *v0, *goal, *x_warm;
    const uint8_t *has_goal;
    double *x, *cost, *acc, *att, *rates, *thrust;
    int32_t *nit, *nfev, *status, *task;
    double flops;
    int rc;
    const orc_grid *grid;
    double w_obs, free_level;
} batch_job;

static void *batch_worker(void *arg)
{
    batch_job *j = (batch_job *)arg;
    const int N = j->p->horizon, n = 9 * N;
    double *buf = (double *)malloc(sizeof(double) * (n + 10 * N));
    if (!buf) {
        j->rc = -1;
        return NULL;
    }
    double *x = buf, *acc = buf + n, *att = acc + 3 * N, *rates = att + 3 * N,
           *thrust = rates + 3 * N;
    j->flops = 0.0;
    for (int64_t b = j->b0; b < j->b1; ++b) {
        orc_stats st;
        const double *goal = (j->has_goal && !j->has_goal[b]) ? NULL : j->goal + 3 * b;
        const double *xw = j->x_warm ? j->x_warm + (int64_t)n * b : NULL;
        int rc = solve_impl(j->p, j->p0 + 3 * b, j->v0 + 3 * b, goal, xw, x, acc, att, rates, thrust,
                            &st, j->grid, j->w_obs, j->free_level);
        if (rc) j->rc = rc;
        j->flops += st.flops;
        if (j->x) memcpy(j->x + (int64_t)n * b, x, sizeof(double) * n);
        if (j->cost) j->cost[b] = st.f;
        if (j->nit) j->nit[b] = st.nit;
        if (j->nfev) j->nfev[b] = st.nfev;
        if (j->status) j->status[b] = st.status;
        if (j->task) j->task[b] = st.task;
        if (j->acc) memcpy(j->acc + (int64_t)3 * N * b, acc, sizeof(double) * 3 * N);
        if (j->att) memcpy(j->att + (int64_t)3 * N * b, att, sizeof(double) * 3 * N);
        if (j->rates) memcpy(j->rates + (int64_t)3 * N * b, rates, sizeof(double) * 3 * N);
        if (j->thrust) memcpy(j->thrust + (int64_t)N * b, thrust, sizeof(double) * N);
    }
    free(buf);
    return NULL;
}

int orc_solve_batch(const orc_params *p, int64_t B, const double *p0, const double *v0,
                    const double *goal, const uint8_t *has_goal, const double *x_warm,
                    double *x, double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                    int32_t *task, double *acc, double *att, double *rates, double *thrust,
                    double *flops_total, int nthreads)
{
    return orc_solve_batch_grid(p, B, p0, v0, goal, has_goal, x_warm, x, cost, nit, nfev, status, task,
                                acc, att, rates, thrust, flops_total, nthreads, NULL, 0.0, 0.0);
}

int orc_solve_batch_grid(const orc_params *p, int64_t B, const double *p0, const double *v0,
                         const double *goal, const uint8_t *has_goal, const double *x_warm,
                         double *x, double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                         int32_t *task, double *acc, double *att, double *rates, double *thrust,
                         double *flops_total, int nthreads, const orc_grid *grid, double w_obs,
                         double free_level)
{
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    if ((int64_t)nthreads > B) nthreads = B > 0 ? (int)B : 1;
    batch_job *jobs = (batch_job *)calloc(nthreads, sizeof(batch_job));
    pthread_t *th = (pthread_t *)calloc(nthreads, sizeof(pthread_t));
    if (!jobs || !th) {
        free(jobs);
        free(th);
        return -1;
    }
    int rc = 0;
    for (int t = 0; t < nthreads; ++t) {
        batch_job *j = &jobs[t];
        j->p = p;
        j->b0 = B * t / nthreads;
        j->b1 = B * (t + 1) / nthreads;
        j->p0 = p0; j->v0 = v0; j->goal = goal; j->x_warm = x_warm; j->has_goal = has_goal;
        j->x = x; j->cost = cost; j->acc = acc; j->att = att; j->rates = rates; j->thrust = thrust;
        j->nit = nit; j->nfev = nfev; j->status = status; j->task = task;
        j->grid = grid; j->w_obs = w_obs; j->free_level = free_level;
        if (nthreads == 1)
            batch_worker(j);
        else if (pthread_create(&th[t], NULL, batch_worker, j) != 0) {
            batch_worker(j);
            th[t] = 0;
        }
    }
    double fl = 0.0;
    for (int t = 0; t < nthreads; ++t) {
        if (nthreads > 1 && th[t]) pthread_join(th[t], NULL);
        fl += jobs[t].flops;
        if (jobs[t].rc) rc = jobs[t].rc;
    }
    if (flops_total) *flops_total = fl;
    free(jobs);
    free(th);
    return rc;
}

/* ======================= mapper (explicit_geometric_mapper.py) ======================= */

/* :91-94 world_to_voxel = floor(p / res) */
void orc_world_to_voxel(double res, const double *p, int32_t *key)
{
    for (int c = 0; c < 3; ++c) key[c] = (int32_t)floor(p[c] / res);
}

static double grid_at(const orc_grid *g, const int32_t *key)
{
    int ix = key[0] - g->ox, iy = key[1] - g->oy, iz = key[2] - g->oz;
    if (ix < 0 || iy < 0 || iz < 0 || ix >= g->nx || iy >= g->ny || iz >= g->nz) return g->prior;
    return (double)g->occ[((int64_t)iz * g->ny + iy) * g->nx + ix];
}

/* :154-169 query_occupancy (dict miss -> prior) */
double orc_query(const orc_grid *g, const double *p)
{
    int32_t key[3];
    orc_world_to_voxel(g->resolution, p, key);
    return grid_at(g, key);
}

/* :195-219 is_trajectory_safe with the :338-351 stencil (centre, -x,+x,-y,+y,-z,+z) */
int orc_traj_safe(const orc_grid *g, const double *positions, int npos, double margin,
                  double threshold)
{
    for (int i = 0; i < npos; ++i) {
        const double *c = positions + 3 * i;
        if (orc_query(g, c) > threshold) return i;
        for (int axis = 0; axis < 3; ++axis)
            for (int dir = -1; dir <= 1; dir += 2) {
                double q[3] = {c[0], c[1], c[2]};
                q[axis] = c[axis] + dir * margin;
                if (orc_query(g, q) > threshold) return i;
            }
    }
    return -1;
}

/* :250-309 _trace_ray */
int orc_trace_ray(double res, const double *start, const double *dir_in, double distance,
                  int32_t *voxels, int max_vox)
{
    double nrm = sqrt(dir_in[0] * dir_in[0] + dir_in[1] * dir_in[1] + dir_in[2] * dir_in[2]);
    double dir[3], end[3], t_delta[3], t_max[3];
    int32_t cur[3], endv[3], step[3];
    for (int c = 0; c < 3; ++c) {
        dir[c] = dir_in[c] / nrm;
        end[c] = start[c] + dir[c] * distance;
    }
    orc_world_to_voxel(res, start, cur);
    orc_world_to_voxel(res, end, endv);
    int count = 0;
    if (count < max_vox) memcpy(voxels + 3 * count, cur, sizeof(cur));
    count++;
    for (int c = 0; c < 3; ++c) {
        step[c] = endv[c] > cur[c] ? 1 : (endv[c] < cur[c] ? -1 : 0);
        if (step[c] != 0) {
            t_delta[c] = res / fabs(dir[c]);
            double boundary = (double)(cur[c] + (step[c] > 0 ? 1 : 0)) * res;
            t_max[c] = fabs((boundary - start[c]) / dir[c]);
        } else {
            t_delta[c] = INFINITY;
            t_max[c] = INFINITY;
        }
    }
    double total = 0.0;
    while ((cur[0] != endv[0] || cur[1] != endv[1] || cur[2] != endv[2]) && total <= distance) {
        int axis = 0;
        if (t_max[1] < t_max[axis]) axis = 1;
        if (t_max[2] < t_max[axis]) axis = 2;
        cur[axis] += step[axis];
        total = t_max[axis];
        t_max[axis] += t_delta[axis];
        if (count < max_vox) memcpy(voxels + 3 * count, cur, sizeof(cur));
        count++;
        if (count > (1 << 24)) break; /* NaN guard */
    }
    return count;
}

/* :399-423 add_obstacle: voxel *corner* distance test */
int orc_add_sphere(orc_grid *g, const double *center, double radius, float value)
{
    int32_t vc[3];
    orc_world_to_voxel(g->resolution, center, vc);
    int vr = (int)ceil(radius / g->resolution);
    int nset = 0;
    for (int dx = -vr; dx <= vr; ++dx)
        for (int dy = -vr; dy <= vr; ++dy)
            for (int dz = -vr; dz <= vr; ++dz) {
                int32_t key[3] = {vc[0] + dx, vc[1] + dy, vc[2] + dz};
                double wx = key[0] * g->resolution - center[0];
                double wy = key[1] * g->resolution - center[1];
                double wz = key[2] * g->resolution - center[2];
                double dist = sqrt(wx * wx + wy * wy + wz * wz);
                if (dist <= radius) {
                    nset++;
                    int ix = key[0] - g->ox, iy = key[1] - g->oy, iz = key[2] - g->oz;
                    if (ix < 0 || iy < 0 || iz < 0 || ix >= g->nx || iy >= g->ny || iz >= g->nz)
                        continue;
                    g->occ[((int64_t)iz * g->ny + iy) * g->nx + ix] = value;
                }
            }
    return nset;
}

/* :311-336 _bayesian_update (hit likelihood 0.7, miss likelihood 1 - 0.4 = 0.6) */
double orc_bayes(double p, int hit)
{
    double lik = hit ? 0.7 : 1 - 0.4;
    double num = lik * p;
    double den = lik * p + (1 - lik) * (1 - p);
    if (den > 0) p = num / den;
    if (p < 0.01) p = 0.01;
    if (p > 0.99) p = 0.99;
    return p;
}

/* :100-152 update_map, sequential like the reference (observation order, voxel order along the
 * ray).  occ64: [nz][ny][nx] doubles (the reference stores Python floats); counts: per-cell
 * observation_count or NULL.  Voxels outside the dense grid are walked and counted (the
 * reference's dict would create them) but not stored.  hit[i] = NaN means hit_distance=None.
 * Returns `updated_voxels`. */
int64_t orc_update_map(const orc_grid *g, double *occ64, int32_t *counts, int64_t n, const double *pos,
                       const double *dir, const double *hit, const double *obs_max_range,
                       double mapper_max_range)
{
    int64_t updated = 0;
    int cap = 1 << 16;
    int32_t *vox = (int32_t *)malloc(sizeof(int32_t) * 3 * cap);
    if (!vox) return -1;
    for (int64_t i = 0; i < n; ++i) {
        const int none = isnan(hit[i]);
        double hd = (none || hit[i] == 0.0) ? obs_max_range[i] : hit[i]; /* falsy -> max_range (:112) */
        if (mapper_max_range < hd) hd = mapper_max_range;
        int cnt = orc_trace_ray(g->resolution, pos + 3 * i, dir + 3 * i, hd, vox, cap);
        if (cnt > cap) {
            cap = cnt;
            free(vox);
            vox = (int32_t *)malloc(sizeof(int32_t) * 3 * cap);
            if (!vox) return -1;
            cnt = orc_trace_ray(g->resolution, pos + 3 * i, dir + 3 * i, hd, vox, cap);
        }
        for (int k = 0; k < cnt; ++k) {
            const int endpoint = (k == cnt - 1) && !none;
            const int ix = vox[3 * k] - g->ox, iy = vox[3 * k + 1] - g->oy, iz = vox[3 * k + 2] - g->oz;
            updated++;
            if (ix < 0 || iy < 0 || iz < 0 || ix >= g->nx || iy >= g->ny || iz >= g->nz) continue;
            const int64_t idx = ((int64_t)iz * g->ny + iy) * g->nx + ix;
            occ64[idx] = orc_bayes(occ64[idx], endpoint);
            if (counts) counts[idx]++;
        }
    }
    free(vox);
    return updated;
}
