/*
 * dart_se3mpc.h -- C ABI of the B200-native batched SE(3)-MPC solve path.
 *
 * The reference (Pasqui1010/DART-Planner) is pure Python and has no FFI for this path; its
 * seam is the class contract of `SE3MPCPlanner` (src/dart_planner/planning/se3_mpc_planner.py).
 * Every entry point below names the reference interface it stands in for.  All pointers are
 * caller-owned DEVICE memory unless a name ends in `_host`; layouts are batch-major
 * structure-of-arrays: a quantity with C components for B problems is `[C][ld]` with the
 * problem index contiguous (`ld >= B` is the row pitch in elements, so a rank can pass a
 * slice of a larger allocation).  Calls are asynchronous on `cuda_stream` (a cudaStream_t),
 * allocate nothing on the hot path, and return 0 or a negative DART_E_* code; they never
 * throw.  Distinct (buffers, stream) pairs may be used concurrently.
 */
#ifndef DART_SE3MPC_H
#define DART_SE3MPC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DART_SE3MPC_ABI_VERSION 1

enum {
    DART_OK = 0,
    DART_E_BADARG = -1,      /* null pointer / negative size / struct_size mismatch        */
    DART_E_UNSUPPORTED = -2, /* horizon > 64, max_corrections > 10, ...                    */
    DART_E_CUDA = -3,        /* a CUDA runtime call failed; see dart_last_cuda_error()     */
    DART_E_NODEVICE = -4
};

/* Termination codes written to `task` (SciPy task numbers in brackets,
 * scipy/optimize/_lbfgsb_py.py as driven by se3_mpc_planner.py:256-268). */
enum {
    DART_TASK_CONV_PGTOL = 1,   /* [401] projected gradient <= gtol                        */
    DART_TASK_CONV_FTOL = 2,    /* [402] relative reduction of f <= ftol                   */
    DART_TASK_STOP_MAXITER = 3, /* [504] wrapper: n_iterations >= maxiter                  */
    DART_TASK_STOP_MAXFUN = 4,  /* [502] wrapper: nfev > maxfun                            */
    DART_TASK_ABNORMAL = 5      /* ABNORMAL: line search failed with no stored pairs       */
};

/* SE3MPCConfig (se3_mpc_planner.py:36-79) + the planner's hard-wired mass/gravity
 * (:149-151) + SciPy's L-BFGS-B options as the reference passes them (:262-267). */
typedef struct dart_se3mpc_params {
    int32_t struct_size;       /* = sizeof(dart_se3mpc_params)                             */
    int32_t horizon;           /* prediction_horizon N, 1..64                              */
    int32_t max_iterations;    /* maxiter                                                  */
    int32_t max_corrections;   /* SciPy maxcor, 1..10 (SciPy default 10)                   */
    int32_t max_linesearch;    /* SciPy maxls, >= 1 (default 20; 0 is DART_E_BADARG)       */
    int32_t max_fun;           /* SciPy maxfun (default 15000)                             */
    int32_t gradient_mode;     /* 0: reference gradient (:552-580, inconsistent by design) */
                               /* 1: exact gradient of :516-550 (extension, self-oracle)   */
                               /* 2: mode 0 + occupancy-grid obstacle penalty in f and g    */
                               /*    (extension, self-oracle; needs a grid, see _solve_batch_map) */
                               /* 3: dynamics-consistent solve (extension, self-oracle): the   */
                               /*    3N thrusts are the only variables; P and V are the rollout */
                               /*    of the plant model (:430-431, :445-459) from (p0, v0):     */
                               /*    a_k = T_k/m - g e3, P_0 = p0, V_0 = v0,                    */
                               /*    P_{k+1} = (P_k + V_k dt) + (0.5 a_k) dt^2,                 */
                               /*    V_{k+1} = V_k + a_k dt.  f is :516-550 at [P | V | T], g   */
                               /*    its exact gradient in T (adjoint).  The P/V rows of x are  */
                               /*    OUTPUTS (the rollout of the returned T; the P/V rows of a  */
                               /*    warm start are ignored); pos_bound and max_velocity are    */
                               /*    NOT enforced.  Closed-loop step: warm == 2 is refused.     */
                               /*    Horizons 1..16 (DART_E_UNSUPPORTED above).                 */
                               /* 4: mode 3 + the obstacle penalty of mode 2 on the rolled-out  */
                               /*    positions (needs a grid; closed loop: _step_map)           */
                               /* 5: mode 0 + the sphere penalty (dart_spheres) on the position */
                               /*    variables; horizons 1..64 (the _spheres entries only)      */
                               /* 6: mode 3 + the sphere penalty on the rolled-out positions;   */
                               /*    horizons 1..16, warm == 2 refused (the _spheres entries)   */
                               /* 7: mode 3 with a per-timestep reference (dart_track_ref);     */
                               /*    horizons 1..16 (the _track entries only)                   */
                               /* 8: mode 6 with the reference of mode 7 (the _track entries)   */
    int32_t reserved0;
    double dt;                 /* effective planner dt (timing_alignment.py:76-78)         */
    double mass, gravity;      /* 1.5 kg, 9.81 m/s^2 (:149-150)                            */
    double pos_bound;          /* +-100 m (:384)                                           */
    double max_velocity;       /* (:388)                                                   */
    double tilt_thrust;        /* max_thrust*sin(max_tilt_angle) (:393-397)                */
    double min_thrust, max_thrust; /* (:400)                                               */
    double w_pos, w_vel, w_acc, w_thrust; /* cost weights (:56-59)                          */
    double gtol;               /* convergence_tolerance (:264)                             */
    double ftol;               /* 10*convergence_tolerance (:265)                          */
    /* gradient_mode 2 and 4 only: f += w_obstacle * sum_k max(0, o(P_k) - obstacle_free_level)^2 with
     * o = trilinear occupancy over voxel centres.  w_obstacle = SE3MPCConfig.obstacle_weight
     * (:60, unused by the reference solve), free level = the map's prior (0.5). */
    double w_obstacle, obstacle_free_level;
} dart_se3mpc_params;

/* Sphere obstacle list of gradient_mode 5 and 6 (extension; the reference builds the constraint
 * |P_k - c|^2 >= (r + safety_margin)^2, se3_mpc_planner.py:499-514, and never passes it to
 * minimize).  One list serves the whole batch.  With w = params->w_obstacle (obstacle_weight), for
 * every timestep k < N and every sphere j = 0 .. n-1 in list order, each product and sum
 * individually rounded (no contraction):
 *   e  = P_k - c_j                          (per component)
 *   d2 = (e_x*e_x + e_y*e_y) + e_z*e_z
 *   R  = r_j + margin
 *   h  = R*R - d2
 *   if h > 0:  f += w*(h*h);   grad_{P_k} += ((-4*w)*h) * e
 * the quadratic penalty of the reference's constraint function d2 - R^2: no square root, no
 * division, a continuous gradient.  Per timestep the penalty sum starts at +0 and its gradient at
 * -0, so a position no sphere reaches leaves the objective and gradient bits of mode 0 / 3 as they
 * are.  At P_k = c_j the gradient is zero (a stationary point of the penalty).  Mode 5 adds it where
 * mode 2 adds the grid penalty (the position variables), mode 6 where mode 4 does (the rolled-out
 * positions, entering the adjoint through dP). */
typedef struct dart_spheres {
    int32_t n;             /* >= 0 */
    int32_t reserved;
    const double *cxyzr;   /* [n][4]: centre x, y, z, radius (device memory; host memory in the _host entry) */
    double margin;         /* added to every radius: SE3MPCConfig.safety_margin */
} dart_spheres;

/* Per-timestep reference of gradient_mode 7 and 8 (extension: tracking a time-parametrised path).
 * Everything not stated here is as in mode 3 / 6: variables, bounds, rollout, adjoint, stopping
 * rule, the P/V rows of x receiving the rollout, horizons 1..16.
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
 * The block is batch-major like the P/V rows of x, with the batch's row pitch ld. */
typedef struct dart_track_ref {
    int32_t len;          /* T >= 1 samples per problem, spaced params->dt apart */
    int32_t start;        /* s >= 0: timestep k reads sample j = min(s + k, T - 1) */
    const double *rows;   /* [6T][ld] device memory: rows 3j+c = position, 3T+3j+c = velocity of sample j */
} dart_track_ref;

/* Self-test of the solver's in-line fp64 division (reciprocal seed + Newton + residual
 * correction, csrc/se3mpc_core.cuh) against IEEE division on n random operand pairs with
 * magnitudes in 2^[-emax, emax]; *mismatch_dev (device uint64, caller-zeroed) += number of
 * quotients whose bits differ. */
int dart_ddiv_selftest(int64_t n, uint64_t seed, int32_t emax, uint64_t *mismatch_dev,
                       void *cuda_stream);

/* ---- occupancy grid (perception/explicit_geometric_mapper.py) on a dense device grid ----
 * occ: [nz][ny][nx] (x fastest) of float32 (cell_bytes 4 or 0: half the bytes, probabilities to
 * 1e-7) or float64 (cell_bytes 8: the reference's own precision -- its voxels hold Python floats);
 * voxel key (kx,ky,kz) = floor(p/res) lives at index (kx-ox, ky-oy, kz-oz); keys outside the grid
 * read `prior` (the reference's dict miss, :168).  Every entry that reads a grid refuses one with
 * nx, ny or nz < 1, resolution <= 0, a NULL occ or cell_bytes outside {0, 4, 8} (DART_E_BADARG). */
typedef struct dart_grid {
    int32_t nx, ny, nz;
    int32_t ox, oy, oz;
    double resolution;
    double prior;
    const void *occ;
    int32_t cell_bytes;
    int32_t reserved;
} dart_grid;

int dart_abi_version(void);
const char *dart_last_cuda_error(void);

/* Fills `p` with the reference's defaults (SE3MPCConfig dataclass defaults, effective
 * dt = 1/400 s, SciPy option defaults). */
void dart_se3mpc_default_params(dart_se3mpc_params *p);

/*
 * Batched replacement of SE3MPCPlanner._solve_se3_mpc (se3_mpc_planner.py:230-280):
 * initial guess (:282-359), bounds (:378-402), L-BFGS-B on (:516-550, :552-580), and the
 * solution extraction (:582-654), for B independent problems.
 *
 * inputs   p0, v0, goal : [3][ld]   current position / velocity, goal position
 *          has_goal     : [ld] u8 or NULL (all problems have a goal)           (:341, :523)
 *          x_warm       : [9N][ld] previous solution or NULL (cold start)       (:294-327)
 *          warm_mask    : [ld] u8 or NULL (all warm when x_warm != NULL)
 * outputs  x_out        : [9N][ld]  rows in the reference's packed order [P | V | T] (:361-376)
 *          cost         : [ld]      OptimizeResult.fun
 *          nit,nfev,status,task : [ld] int32 (status as OptimizeResult.status: 0/1/2)
 *          acc, att, rates : [3N][ld] rows 3k+c; thrust : [N][ld]                (:582-654)
 *          any output pointer may be NULL (not written).
 */
int dart_se3mpc_solve_batch(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                            const double *p0, const double *v0, const double *goal,
                            const uint8_t *has_goal, const double *x_warm,
                            const uint8_t *warm_mask, double *x_out, double *cost, int32_t *nit,
                            int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                            double *att, double *rates, double *thrust, void *cuda_stream);

/* Solve + fused post-hoc safety check: the same solve, then `is_trajectory_safe`
 * (explicit_geometric_mapper.py:195-219; as the callers use it after planning,
 * cloud/main_improved_se3.py:128-130) on the N solved positions of every problem, inside the
 * solve kernel (positions never leave registers).  first_hit [ld] int32: index of the first
 * colliding position, -1 = safe.  grid/first_hit may be NULL (plain solve).
 * With params->gradient_mode == 2 the same grid also feeds the obstacle penalty inside the
 * solve (then `grid` is required; first_hit stays optional). */
int dart_se3mpc_solve_batch_map(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                const double *p0, const double *v0, const double *goal,
                                const uint8_t *has_goal, const double *x_warm,
                                const uint8_t *warm_mask, double *x_out, double *cost, int32_t *nit,
                                int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                double *att, double *rates, double *thrust, const dart_grid *grid,
                                double margin, double threshold, int32_t *first_hit,
                                void *cuda_stream);

/* Solution extraction alone: `_extract_solution_from_result` / `_compute_attitudes_and_rates`
 * (se3_mpc_planner.py:582-654) for B given thrust sequences -- the code the solve kernel's epilogue
 * runs, callable with arbitrary thrust vectors.  thrust_vectors: SoA rows 3k+c (k = step,
 * c = x/y/z) of pitch ld; outputs as in dart_se3mpc_solve_batch.  A step with |T| <= 1e-6 gets zero
 * attitude and rates and does not advance the reference's prev_R (:617, :647-651).
 * untilted != 0: the caller promises T_x = T_y = 0 at every step (what a cold-started solve
 * produces); the 7-slot instantiation's extraction runs (closed form when every T_z > 1e-6). */
int dart_se3mpc_extract_batch(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                              const double *thrust_vectors, double *acc, double *att, double *rates,
                              double *thrust, int32_t untilted, void *cuda_stream);

/* Row output: the same solve (and, with check_map != 0, the same fused safety check), with every
 * problem's whole result written as ONE contiguous row -- the arrays the reference packs into
 * the Trajectory it returns for one solve (se3_mpc_planner.py:656-675, from :582-654) next to
 * the OptimizeResult fields it reads (:268-280):
 *   double [0, 9N) x  (reference packed order [P | V | T], :361-376) | [9N] cost |
 *   acc 3N | att 3N | rates 3N (entries 3k+c) | thrust N |
 *   then int32 nit, nfev, status, task, first_hit (-1 safe, -2 not checked), 0
 * i.e. 19N+4 doubles, padded with zeros to `row_stride` doubles.  row_stride must be a multiple
 * of 16 (whole 128-byte lines), >= dart_se3mpc_row_stride(params), and `rows` 128-byte aligned.
 * The kernel stages a row in shared memory and writes it with full-line 16-byte stores, so
 * `rows` -- like p0/v0/goal/has_goal/x_warm -- may be mapped pinned HOST memory: the solve then
 * needs no copy in either direction (the e2e path of BatchWorkspace.solve_rows, bench.py).
 * row_kind 1 (DART_ROWS_CONTROLS): only what a caller forwarding thrust commands needs --
 *   double [0, 3N) T (rows 6N..9N of x: the thrust vectors, :361-376) | [3N] cost |
 *   the same six int32 (first_hit = -2) -- 3N+4 doubles (256 B instead of 1 280 B at N = 8);
 *   no solution extraction is computed, check_map must be 0.
 * row_kind 2 (DART_ROWS_SOLUTION): what scipy.optimize.minimize itself returns (:256-268) --
 *   double [0, 9N) x | [9N] cost | the same six int32 -- 9N+4 doubles (640 B instead of
 *   1 280 B at N = 8).  The derived arrays of :582-654 (acceleration, attitude, body rate,
 *   thrust magnitude) are pure functions of the thrust rows of x and dt and are left to the
 *   caller (dart_planner_b200.planner.HostSolution derives them on first access); the fused
 *   map check is available.
 * dart_se3mpc_row_stride returns the minimal stride for the row kind, or 0 when this horizon's
 * row does not fit the staging block (full rows: N > 25): use the SoA entries then. */
#define DART_ROWS_FULL 0
#define DART_ROWS_CONTROLS 1
#define DART_ROWS_SOLUTION 2
int64_t dart_se3mpc_row_stride(const dart_se3mpc_params *params, int32_t row_kind);
int dart_se3mpc_solve_batch_rows(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                 const double *p0, const double *v0, const double *goal,
                                 const uint8_t *has_goal, const double *x_warm,
                                 const uint8_t *warm_mask, double *rows, int64_t row_stride,
                                 int32_t row_kind, const dart_grid *grid, double margin,
                                 double threshold, int32_t check_map, void *cuda_stream);

/* One replanning step of the closed-loop receding-horizon simulation (BASELINE configs[4]),
 * one launch: solve every problem from its resident state (p, v) -- cold start when warm == 0,
 * else the warm start of se3_mpc_planner.py:294-327 from the previous solution held in x --
 * write the new solution to x, then advance the state in place with the planner's own model
 * (:430-431, :445-459) driven by the first control:  a = T_0/m - g e3,
 * p <- p + v*dt + 0.5*a*dt^2,  v <- v + a*dt  (dt = plant_dt).
 * p, v : [3][ld] in/out;  x : [9N][ld] in/out;  cost/nit/nfev/status may be NULL.
 * warm == 2: warm start with the caller's promise that every lateral thrust entry (T_x, T_y) of
 * x is exactly zero -- true for solutions this library produced from cold starts, since a zero
 * lateral thrust has a zero gradient and never moves.  The faster 7-slot kernel then serves the
 * warm start; a problem whose x breaks the promise is not solved and gets status 3.
 * gradient_mode 3: warm == 2 returns DART_E_BADARG (the lateral thrust moves); with
 * plant_dt == params->dt the new state is the solution's P_1 / V_1.  gradient_mode 2 and 4
 * (obstacle penalty: no map argument here; see dart_se3mpc_closed_loop_step_map) return
 * DART_E_UNSUPPORTED. */
int dart_se3mpc_closed_loop_step(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                 double *v, const double *goal, const uint8_t *has_goal, double *x,
                                 int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                 int32_t *status, double plant_dt, void *cuda_stream);

/* The same step against a map (extension), still one launch:
 *   penalty_grid : the grid of the obstacle penalty, required for gradient_mode 2 and 4 (else
 *                  DART_E_BADARG) and ignored otherwise -- typically a clearance field
 *                  (dart_map_clearance_field) with params->obstacle_free_level = its prior;
 *   check_grid, first_collision : optional together (one without the other: DART_E_BADARG).
 *                  After the plant step, the path of this step from p to p' is sampled at
 *                  q_j = p + (p' - p) * (j / S), j = 1..S, S = max(1, ceil(|p' - p|_inf / (0.5 res)))
 *                  capped at 64 (res = check_grid->resolution; every operation individually
 *                  rounded), and each q_j is tested with is_trajectory_safe's stencil (margin,
 *                  threshold, as in dart_map_traj_safe_batch).  A problem whose path collides and
 *                  whose first_collision [ld] int32 entry is -1 gets `step` there (the caller
 *                  initialises the entries to -1 and passes its step counter).
 * warm == 2 is refused (DART_E_BADARG) in gradient_mode 3 and 4.  Everything else as
 * dart_se3mpc_closed_loop_step; with neither grid the results are the same bits. */
int dart_se3mpc_closed_loop_step_map(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                     double *p, double *v, const double *goal,
                                     const uint8_t *has_goal, double *x, int32_t warm, double *cost,
                                     int32_t *nit, int32_t *nfev, int32_t *status, double plant_dt,
                                     const dart_grid *penalty_grid, const dart_grid *check_grid,
                                     double margin, double threshold, int32_t step,
                                     int32_t *first_collision, void *cuda_stream);

/* ---- the sphere penalty (gradient_mode 5 / 6, see dart_spheres) ------------------------------
 * Every other entry returns DART_E_UNSUPPORTED for gradient_mode 5 and 6.  These three refuse with
 * DART_E_BADARG a gradient_mode other than 5 or 6, a NULL `spheres`, spheres->n < 0, n > 0 with a
 * NULL cxyzr, and warm == 2 in mode 6; mode 6 above horizon 16 is DART_E_UNSUPPORTED.  n == 0 is
 * allowed and returns the bits of mode 0 / 3.  No row-output entry takes spheres.
 *
 * dart_se3mpc_solve_batch_spheres: dart_se3mpc_solve_batch_map with the sphere penalty in the
 * solve; `grid` (with margin, threshold, first_hit) serves only the optional fused safety check. */
int dart_se3mpc_solve_batch_spheres(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                    const double *p0, const double *v0, const double *goal,
                                    const uint8_t *has_goal, const double *x_warm,
                                    const uint8_t *warm_mask, double *x_out, double *cost, int32_t *nit,
                                    int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                    double *att, double *rates, double *thrust, const dart_spheres *spheres,
                                    const dart_grid *grid, double margin, double threshold,
                                    int32_t *first_hit, void *cuda_stream);
/* dart_se3mpc_closed_loop_step_map with the sphere penalty; check_grid / first_collision as there
 * (the collision record against a map, typically the same spheres rasterised by add_obstacles).
 * warm == 2 is allowed in mode 5: its lateral thrust stays exactly zero, as in mode 0. */
int dart_se3mpc_closed_loop_step_spheres(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                         double *p, double *v, const double *goal,
                                         const uint8_t *has_goal, double *x, int32_t warm, double *cost,
                                         int32_t *nit, int32_t *nfev, int32_t *status, double plant_dt,
                                         const dart_spheres *spheres, const dart_grid *check_grid,
                                         double margin, double threshold, int32_t step,
                                         int32_t *first_collision, void *cuda_stream);

/* ---- reference tracking (gradient_mode 7 / 8, see dart_track_ref) ----------------------------
 * Every other entry refuses gradient_mode 7 and 8.  These two return DART_E_BADARG for a
 * gradient_mode other than 7 or 8, a NULL `ref` or ref->rows, ref->len < 1, ref->start < 0, mode 7
 * with spheres or mode 8 without them (dart_spheres as in the _spheres entries; n == 0 gives mode 7's
 * bits), warm == 2, and in the closed-loop step plant_dt != params->dt.  A horizon above 16 is
 * DART_E_UNSUPPORTED.  No host-memory or row-output entry takes a reference.
 *
 * dart_se3mpc_solve_batch_track: dart_se3mpc_solve_batch_spheres without `goal`, with the
 * reference; `grid` (with margin, threshold, first_hit) serves only the optional fused safety check.
 * plan_batch passes T = N and s = 0. */
int dart_se3mpc_solve_batch_track(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                  const double *p0, const double *v0, const uint8_t *has_goal,
                                  const double *x_warm, const uint8_t *warm_mask, double *x_out, double *cost,
                                  int32_t *nit, int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                  double *att, double *rates, double *thrust, const dart_track_ref *ref,
                                  const dart_spheres *spheres, const dart_grid *grid, double margin,
                                  double threshold, int32_t *first_hit, void *cuda_stream);
/* dart_se3mpc_closed_loop_step_spheres without `goal`, with the reference: a path of T samples and
 * s = the step index, so the window slides one sample per replan (plant_dt == params->dt); past the
 * end of the path the last sample is held.  check_grid / first_collision as in the _map step. */
int dart_se3mpc_closed_loop_step_track(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                       double *p, double *v, const uint8_t *has_goal, double *x,
                                       int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                       int32_t *status, double plant_dt, const dart_track_ref *ref,
                                       const dart_spheres *spheres, const dart_grid *check_grid,
                                       double margin, double threshold, int32_t step,
                                       int32_t *first_collision, void *cuda_stream);

/* ---- the differentiable solve: vector-Jacobian product of a returned plan (extension) ---------
 * Scope: gradient_mode 3, 6, 7 and 8, horizons 1..16.  T* is the thrust rows of a returned solution x
 * (any x: the P/V rows are not read).  The bounds l <= T <= u are the solve's own boxes (+-tilt_thrust
 * on x and y, min_thrust..max_thrust on z).  The active set A is the set of entries with T*_i == l_i
 * or T*_i == u_i, bit for bit (L-BFGS-B projects onto the box exactly); F is every other entry.
 * Parameters theta, per problem: p0 and v0; the goal (modes 3 / 6) or the reference r_k, u_k (modes
 * 7 / 8); the weights w = (w_pos, w_vel, w_acc, w_thrust).  The derivative holds T*_A constant and
 * takes dT*_F/dtheta = -H_FF^-1 dg_F/dtheta, with g = grad_T f and H = hess_T f at the returned T*:
 * defined at whatever T* the solve returned, converged or not.  (In modes 3 / 7, H and the derivatives
 * with respect to p0, v0, goal and reference do not depend on T*; the weight derivatives do, as dg/dw
 * is linear in T.)  Outputs that carry a derivative: x = [P | V | T], where P and V are the rollout of
 * T*(theta) from (p0, v0), P_0 = p0 and V_0 = v0 included; and cost = f(T*(theta), theta).
 * Given upstream gradients xbar (9N) and cbar (one per problem), the entry:
 *   1. pulls xbar back through the rollout with the solve's adjoint,
 *   2. adds cbar g(T*),
 *   3. solves H_FF lam_F = tbar_F with lam_A = 0 (matrix-free conjugate gradients on F; every Hessian
 *      product is a zero-state rollout and one adjoint; n_F <= 3N steps in exact arithmetic),
 *   4. forms thetabar = -(dg/dtheta)^T lam + cbar df/dtheta + the rollout's direct dependence on p0 and
 *      v0; (dg/dtheta)^T lam comes from one forward rollout of lam from a zero state.
 * Modes 6 and 8 add the sphere penalty's Hessian on P_k where h > 0, 8 w e e^T - 4 w h I in the
 * notation of dart_spheres; H_FF can then be indefinite.
 * status [ld] per problem: 0 ok; 1 non-positive curvature met; 2 the linear solve did not reach its
 * residual tolerance (|r| <= 1e-13 |tbar_F| within 2 n_F + 8 products).  Status 1 is a property of the
 * system solved for this problem's upstream gradients, not of H_FF alone: conjugate gradients meet the
 * curvature of H_FF only along the directions tbar_F reaches.  Where tbar_F is exactly zero no step runs,
 * lam = 0 and the status is 0 even if H_FF is indefinite (the returned gradients are then exact).  Where
 * the status is not 0, every gradient output of that problem is NaN.
 *
 * inputs   params, p0, v0, goal, has_goal : as in the solve that returned x (goal: modes 3 / 6 only,
 *          not read in 7 / 8 or where has_goal is 0); ref (modes 7 / 8) with len = N and start = 0, as
 *          plan_batch passes it; spheres (modes 6 / 8) as in the solve
 *          x  : [9N][ld] the solve's solution
 *          gx : [9N][ld] xbar, gcost : [ld] cbar; either may be NULL (zero)
 * outputs  gp0, gv0 : [3][ld];  ggoal : [3][ld] (modes 3 / 6; not written in 7 / 8);
 *          gref : [6N][ld] in the layout of the reference block (rows 3k+c rbar_k, 3N+3k+c ubar_k;
 *          modes 7 / 8; not written in 3 / 6);  gw : [4][ld] wbar per problem;  any may be NULL
 *          status : [ld] int32, required
 * Refused with DART_E_BADARG: a gradient_mode outside {3, 6, 7, 8}; spheres in modes 3 / 7 or none in
 * 6 / 8 (n < 0, or n > 0 with a NULL list); a reference in modes 3 / 6 or none in 7 / 8; ref->len != N,
 * ref->start != 0 or a NULL ref->rows; NULL x, status, p0, v0, or goal in modes 3 / 6; B < 0 or
 * ld < B.  A horizon above 16 is DART_E_UNSUPPORTED.  No gradient flows to warm starts, sphere
 * centres or radii, obstacle_weight, or the derived arrays (attitudes, rates). */
int dart_se3mpc_solve_vjp_batch(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                const double *p0, const double *v0, const double *goal,
                                const uint8_t *has_goal, const double *x, const dart_track_ref *ref,
                                const dart_spheres *spheres, const double *gx, const double *gcost,
                                double *gp0, double *gv0, double *ggoal, double *gref, double *gw,
                                int32_t *status, void *cuda_stream);

/* Same call with every buffer in HOST memory (pageable or pinned).  Up to 512 problems go
 * through a mapped pinned block the kernel reads and writes directly (no copies); larger batches
 * stage through an internal per-thread device workspace (chunked on two streams from 65536
 * problems up).  Returns after synchronising.
 * This is the plugin-level entry the drop-in planner's single-problem `plan()` uses. */
int dart_se3mpc_solve_batch_host(const dart_se3mpc_params *params, int64_t B,
                                 const double *p0_host, const double *v0_host,
                                 const double *goal_host, const uint8_t *has_goal_host,
                                 const double *x_warm_host, double *x_out_host,
                                 double *cost_host, int32_t *nit_host, int32_t *nfev_host,
                                 int32_t *status_host, double *acc_host, double *att_host,
                                 double *rates_host, double *thrust_host);

/* dart_se3mpc_solve_batch_host with the sphere penalty; spheres->cxyzr is HOST memory, staged with
 * the other inputs (the mapped block up to 512 problems, the device workspace above). */
int dart_se3mpc_solve_batch_host_spheres(const dart_se3mpc_params *params, int64_t B,
                                         const double *p0_host, const double *v0_host,
                                         const double *goal_host, const uint8_t *has_goal_host,
                                         const double *x_warm_host, double *x_out_host,
                                         double *cost_host, int32_t *nit_host, int32_t *nfev_host,
                                         int32_t *status_host, double *acc_host, double *att_host,
                                         double *rates_host, double *thrust_host,
                                         const dart_spheres *spheres);

/* Frees what dart_se3mpc_solve_batch_host caches for the CALLING thread (device workspace, mapped
 * pinned staging block, two streams) after draining them.  A host thread that used the host
 * entry calls this before it exits; the next call of the host entry allocates again. */
void dart_se3mpc_release_thread_workspace(void);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t dart_launch_count(void);

/* A caller that keeps several launches in flight on different streams (a stream of planning
 * steps, each a batch of its own) says how many problems that is in total: the build is then
 * chosen for that number instead of one launch's B -- four 4 096-problem steps in flight fill the
 * machine like one 16 384-problem launch, and the register-capped throughput build (3 resident
 * blocks per SM) serves them at 14.4 us per step where one step at a time takes 24.7 us in the
 * latency build.  0 restores the per-launch choice.  Process-wide; row-output launches always use
 * the latency build.  (No counterpart in the reference: its planner solves one problem per call,
 * se3_mpc_planner.py:215-228.) */
int dart_se3mpc_set_inflight_hint(int64_t problems_in_flight);

/* Name, registers and launch geometry of the solve kernel chosen for (horizon, B). */
int dart_se3mpc_kernel_info(const dart_se3mpc_params *params, int64_t B, int32_t *lanes,
                            int32_t *block_threads, int32_t *grid_blocks, int32_t *smem_bytes,
                            int32_t *regs_per_thread);

/* FP64 FMA throughput probe (bench.py's compute-roofline denominator): launches
 * 148*8 blocks x 256 threads, each running 8 independent DFMA chains of `iters` steps;
 * flops = threads * 8 * iters * 2.  `scratch`: >= 8 bytes of device memory. */
int dart_fp64_probe(int32_t iters, int32_t *threads_out, double *scratch, void *cuda_stream);

/* query_occupancy_batch (:171-182): pos [3][ld] -> occ_out [ld] (float64 like the reference) */
int dart_map_query_batch(const dart_grid *g, int64_t B, int64_t ld, const double *pos,
                         double *occ_out, void *cuda_stream);
/* is_trajectory_safe (:195-219, stencil :338-351) for B trajectories of npos points:
 * positions [3*npos][ld] rows 3k+c  ->  first_hit [ld] int32 (-1 = safe) */
int dart_map_traj_safe_batch(const dart_grid *g, int64_t B, int64_t ld, int32_t npos,
                             const double *positions, double margin, double threshold,
                             int32_t *first_hit, void *cuda_stream);
/* _trace_ray (:250-309) for B rays: start, dir [3][ld], dist [ld] -> count [ld] voxels
 * visited; if voxels != NULL the first min(count,max_vox) keys are written to
 * voxels [max_vox][3][ld] int32. */
int dart_map_trace_ray_batch(double resolution, int64_t B, int64_t ld, const double *start,
                             const double *dir, const double *dist, int32_t max_vox,
                             int32_t *count, int32_t *voxels, void *cuda_stream);
/* update_map (:100-152) for a scan of B observations (SensorObservation :40-47): start, dir
 * [3][ld]; hit_distance [ld] (NaN = None: no return); obs_max_range [ld] (the observation's own
 * max_range, used when hit_distance is falsy :112); mapper_max_range caps the ray (:113).
 * Every voxel on a ray gets a Bayes "miss" update, the last one a "hit" update when there was a
 * return (:118-135), with likelihoods prob_hit and 1 - prob_miss (:322-327) and the clip to
 * [0.01, 0.99].  counts: caller-owned scratch of nx*ny*nz uint64, zero on entry, zero on return.
 * updated_voxels: optional device counter, incremented by the number of voxel visits (the
 * reference's `updated_voxels`).  Voxels outside the dense grid are visited but not stored. */
int dart_map_update_batch(const dart_grid *g, void *occ_writable, uint64_t *counts, int64_t B,
                          int64_t ld, const double *start, const double *dir,
                          const double *hit_distance, const double *obs_max_range,
                          double mapper_max_range, double prob_hit, double prob_miss,
                          uint64_t *updated_voxels, void *cuda_stream);
/* add_obstacle (:399-423): rasterise n spheres (centres [3][n], radii [n]) into a writable
 * grid with the reference's voxel-corner distance test; value 0.9. */
int dart_map_add_spheres(const dart_grid *g, void *occ_writable, int32_t n,
                         const double *centers, const double *radii, double value,
                         void *cuda_stream);

/* ---- signed distance and clearance field of a grid (extension; the reference has none) ----
 * Occupied means occ > threshold (is_collision's strict test).  For every cell, D+ is the squared
 * distance in voxels from its centre to the nearest occupied cell centre and D- the same to the
 * nearest free cell centre, both exact integers (separable lower envelope of parabolas,
 * Felzenszwalb-Huttenlocher, integer comparisons only; three launches, x, y, z).  Only cells of
 * the box are sites: with no occupied cell D+ is the squared box diagonal nx^2+ny^2+nz^2, with no
 * free cell D- is.
 *   phi = res * (sqrt(D+) - sqrt(D-))   [m, float32, rounded once from double]
 * sq_scratch: 2*nx*ny*nz int32 of device memory.  On return its first nx*ny*nz entries hold the
 * signed squared distance: D+ at a free cell, -D- at an occupied cell (the other one is 0).
 * phi_out: nx*ny*nz float32 in the grid's cell order, or NULL (then only sq_scratch is written).
 * DART_E_UNSUPPORTED when nx^2+ny^2+nz^2 >= 2^30 - 1. */
int dart_map_signed_distance(const dart_grid *g, double threshold, float *phi_out,
                             int32_t *sq_scratch, void *cuda_stream);
/* Clearance field for the obstacle penalty of gradient_mode 2 / 4: the same transform, then
 *   c = free_level + max(0, safety_distance - phi)    (double, from the float32 phi)
 * stored in the grid's own cell type (cell_bytes) to field_out (nx*ny*nz cells, same order).  Used
 * as a penalty grid with prior = obstacle_free_level = free_level, a cell farther than
 * safety_distance from every occupied cell (and every key outside the box) costs nothing and
 * gives no gradient; inside an obstacle the field keeps rising with the depth.  sq_scratch as
 * above (and holding the same result on return). */
int dart_map_clearance_field(const dart_grid *g, double threshold, double safety_distance,
                             double free_level, void *field_out, int32_t *sq_scratch,
                             void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* DART_SE3MPC_H */
