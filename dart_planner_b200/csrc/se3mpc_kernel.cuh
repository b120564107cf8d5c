/*
 * se3mpc_kernel.cuh -- the solve kernel template (one problem per sub-warp, see se3mpc_core.cuh)
 * and the per-configuration table its instantiation units export.  Each lane configuration is
 * compiled in its own translation unit (se3mpc_inst_*.cu) so the build runs in parallel.
 *
 * Replaces: SE3MPCPlanner._solve_se3_mpc (se3_mpc_planner.py:230-280) for B problems.
 */
#pragma once
#include <cuda_runtime.h>

#include <utility>

#include "map_query.cuh"
#include "se3mpc_core.cuh"

namespace dartb200 {

struct SolveArgs {
    long long B, ld;
    const double *p0, *v0, *goal;
    const unsigned char *has_goal;
    const double *x_warm;
    const unsigned char *warm_mask;
    double *x_out, *cost;
    int *nit, *nfev, *status, *task;
    double *acc, *att, *rates, *thrust;
    /* the obstacle penalty's grid (gradient_mode 2 / 4) */
    dart_grid grid;
    /* fused post-solve safety check (is_trajectory_safe on the solved positions) against
     * check_grid; on when check_map != 0.  The same grid as `grid` except in the closed-loop step
     * with a map, whose penalty grid and collision map are separate */
    dart_grid check_grid;
    double margin, threshold;
    int *first_hit;
    int check_map; /* 1: run the check (SoA mode: into first_hit; row mode: into the row) */
    /* fused plant step of the closed-loop simulation (off when p_next == nullptr): the state is
     * advanced with the first control of the new solution; may alias p0 / v0 */
    double *p_next, *v_next;
    double plant_dt;
    /* collision record of the plant step (off when first_collision == nullptr): the step's path
     * p -> p_next, sampled at most half a voxel apart, against check_grid (margin, threshold);
     * a problem whose path collides and whose first_collision is -1 gets `step` */
    int *first_collision;
    int step;
    /* the caller promises that every lateral thrust entry of x_warm is exactly zero (solutions
     * this library produced from cold starts): the 7-slot instantiation then serves warm starts
     * too.  The kernel checks the promise per problem and refuses (status 3) where it is broken. */
    int no_tilt_promise;
    /* row output (off when rows == nullptr): every problem's whole result is ONE contiguous row
     *   [x 9N | cost | acc 3N | att 3N | rates 3N | thrust N | int32 nit nfev status task first_hit 0]
     * of row_stride doubles (a multiple of 16: whole 128-byte lines), staged in the problem's
     * shared block and written with 16-byte stores, lane after lane -- the access pattern that
     * lets `rows` be pinned HOST memory (zero-copy over PCIe) at close to the link rate.  The
     * SoA output pointers above are ignored in this mode (the map check's result goes into the
     * row). */
    double *rows;
    long long row_stride;
    /* 0: the full row above; 2: solution row [x 9N | cost | the int32 block] (the derived arrays
     * left out: 9N+4 doubles, 640 B at N=8); 1: controls row [T 3N (rows 6N..9N of x) | cost | the same int32
     * block with first_hit = -2] for callers that only forward the thrust commands: 3N+4 doubles
     * (256 B at N=8 instead of 1 280 B over PCIe), no solution extraction, no map check */
    int rows_kind;
    /* dynamic schedules: queue[0] ticket counter, queue[1] finished blocks; both zero at launch and
     * re-armed by the last block of the launch */
    unsigned long long *queue;
    /* two-phase schedule: context slots, grid x (2 GPB - 1) x ctx_doubles(1) doubles */
    double *stash;
    /* Long solves first (throughput builds, cold starts, large batches; off when prio_count ==
     * nullptr).  A problem that starts within ~1 m of its goal ends in the reference's degenerate
     * line-search regime -- two searches of 20 evaluations, ~4x the serial work of a normal solve
     * -- and a launch lasts until the last of them is done, so one that is handed out late extends
     * the launch by its own length (65 536 problems: 238 vs 304 us, profiles/README.md).  A scan
     * kernel in front of the solve lists the problems with |goal - p0|^2 < prio_r2 (at most
     * PRIO_CAP of them; a longer list, or one longer than B/64, switches the feature off for the
     * launch).  The solve does not wait for the scan: it is launched as a programmatic dependent of
     * it, every block's first round is a regular one, and only a block that comes back for more
     * waits for the scan's completion (long past by then) and reads the list.  Tickets: G = grid
     * size; t < G: regular round t; G <= t < G + P: priority round (members below G*GPB were
     * solved in the first rounds already); later t: regular round t - P, members of the list
     * skipped.  Scheduling only: which sub-warp solves a problem when has no effect on its result.
     * prio_count is reset by the last block of the solve (the slot is reused by a later launch). */
    int *prio_list;
    unsigned *prio_count;
    double prio_r2;
    /* the sphere list of the obstacle penalty (gradient_mode 5 / 6): [n_spheres][4] doubles (cx, cy,
     * cz, r) of device memory, every radius inflated by sphere_margin.  Last, so that the fields
     * above keep their offsets; 0 spheres in every launch of the other modes */
    const double *spheres;
    int n_spheres;
    double sphere_margin;
    /* the per-timestep reference of gradient_mode 7 / 8 (dart_track_ref): [6 track_len][ld] doubles of
     * device memory; timestep k of a solve reads sample min(track_start + k, track_len - 1).  Last,
     * as the sphere fields; null / 0 in every launch of the other modes */
    const double *track_rows;
    int track_len, track_start;
};
constexpr int PRIO_CAP = 16384;

/* member of the priority list?  (the same predicate in the scan kernel and in the solve kernel) */
__device__ __forceinline__ bool starts_near_goal(const SolveArgs &A, long long b)
{
    if (A.has_goal && A.has_goal[b] == 0) return false;
    const double dx = __ldg(A.goal + b) - __ldg(A.p0 + b);
    const double dy = __ldg(A.goal + A.ld + b) - __ldg(A.p0 + A.ld + b);
    const double dz = __ldg(A.goal + 2 * A.ld + b) - __ldg(A.p0 + 2 * A.ld + b);
    return dx * dx + dy * dy + dz * dz < A.prio_r2;
}

__global__ void __launch_bounds__(256) se3mpc_prio_scan_kernel(const __grid_constant__ SolveArgs A);

/* doubles of one result row (before padding) and the padded stride; 0 when the row does not fit
 * the per-problem shared block it is staged in */
__host__ __device__ inline int row_payload_doubles(int N, int kind)
{
    return (kind == 1 ? 3 : (kind == 2 ? 9 : 19)) * N + 4;
}
__host__ __device__ inline int row_stride_doubles(int N, int kind)
{
    const int st = (row_payload_doubles(N, kind) + 15) / 16 * 16;
    return st <= SM_DOUBLES ? st : 0;
}

/* Problems (lane groups) per block and this thread's group.  LANES = 6: five groups per warp, the
 * warp's last two lanes own no problem (`idle`; they follow the block's barriers and the warp's
 * round loop, alias the warp's last group index and never start a solve). */
template <int LANES, int BLOCK>
struct GroupMap {
    static constexpr int GPW = 32 / LANES;
    static constexpr int GPB = (BLOCK / 32) * GPW;
    __device__ static __forceinline__ bool idle() { return (LANES * GPW != 32) && (int)(threadIdx.x & 31) >= LANES * GPW; }
    __device__ static __forceinline__ int gib()
    {
        const int g = (int)(threadIdx.x & 31) / LANES;
        return (int)(threadIdx.x >> 5) * GPW + (g < GPW ? g : GPW - 1);
    }
};

template <int LANES, int TPL, int BLOCK, int MINB, int GM, bool TILT>
__global__ void __launch_bounds__(BLOCK, MINB)
se3mpc_solve_kernel(const __grid_constant__ dart_se3mpc_params P, const __grid_constant__ SolveArgs A)
{
    extern __shared__ double smem_all[];
    using GMap = GroupMap<LANES, BLOCK>;
    constexpr int GPB = GMap::GPB; /* problems (groups) per block */
    const int gib = GMap::gib();
    const bool idle_lane = GMap::idle();
    double *sm = smem_all + gib * SM_DOUBLES;
    const int N = P.horizon;
    double ws[MMAX][9 * TPL], wy[MMAX][9 * TPL]; /* per-lane S / Y pairs (local memory, L1) */
    /* How problems reach the sub-warps.
     *   SCHED 0  static: block b takes rounds b, b + grid, ... of GPB problems (latency builds: one
     *            round, nothing to balance).
     *   SCHED 1  dynamic per warp: a warp takes the next 32/LANES problems from a global ticket
     *            counter when it has finished its own, so no SM idles behind the slowest static share
     *            (65 536 problems: 381 -> 296 us; the solves differ 3x in length; 1 Mi: 4.87 -> 4.57 ms).
     *   SCHED 2  dynamic per block + lock step: the block takes GPB problems per ticket and its
     *            warps start every L-BFGS-B iteration together (one barrier per iteration), so they
     *            run the same straight-line code at the same time and share its instruction fetches
     *            (65 536: 290 us; 1 Mi: 4.18 ms = 251 M solves/s.  Lock step on the static schedule,
     *            SCHED 3, gives 376 us / 4.54 ms; in a single-round latency launch it only adds waiting).
     * The throughput builds use DART_THROUGHPUT_SCHED (profiles/README.md, round 2). */
#ifndef DART_THROUGHPUT_SCHED
#define DART_THROUGHPUT_SCHED 2
#endif
#ifndef DART_LATENCY_SCHED
#define DART_LATENCY_SCHED 0
#endif
    constexpr int SCHED = (MINB >= 3) ? DART_THROUGHPUT_SCHED : DART_LATENCY_SCHED;
    constexpr bool LOCK = (SCHED == 2) || (SCHED == 3);
    using SolverT = Solver<typename GroupOf<LANES>::type, TPL, GM, (MINB >= 3), TILT>;
    /* two-phase schedule (SCHED 4): contexts of the problems between their first iteration and
     * the rest of their solve, GPB - 1 left over + GPB new ones at most, per block, in global
     * memory (L2-resident: written once, read once) */
    constexpr int STASH_CAP = 2 * GPB - 1;
    constexpr int CTXD = SolverT::ctx_doubles(1);
    __shared__ int s_cont[GPB];
    __shared__ int s_stash_n;
    /* one problem, solved by this thread's sub-warp.  `alive` = false (lock-step builds only): a
     * padding sub-warp that solves a copy of the last problem and writes nothing, so that every
     * thread of the block reaches the block barriers.
     * phase 0: the whole solve.  Phases of the two-phase schedule, block-uniform: 1 = a fresh
     * problem's start and FIRST iteration (finished: results out; else its context goes to the
     * block's stash), 2 = a stashed problem (`alive` = this sub-warp has one, taken from slot
     * `b_in`) continues to the end, the block in lock step. */
    auto solve_one = [&](const long long b_in, const bool alive, const int phase, const bool skip_near = false) {
        /* a padding sub-warp (lock-step builds: ragged last round, a skipped member of the priority
         * list) keeps the block's barriers company but starts no solve.  (Starting one and cutting
         * it after the first evaluation, so that `refused` stays a compile-time false in the
         * cold-start kernels, was measured: 1 % slower.) */
        bool refused = !alive || idle_lane;
        long long b = b_in;
        SolverT sv(P, sm, ws, wy);
        if constexpr (SolverT::SPHERES) {
            sv.obs.s = A.spheres;
            sv.obs.n = A.n_spheres;
            sv.obs.w = P.w_obstacle;
            sv.obs.margin = A.sphere_margin;
        } else if constexpr (SolverT::POS_PEN || SolverT::ROLLOUT_PEN) {
            sv.obs.g = A.grid;
            sv.obs.w = P.w_obstacle;
            sv.obs.free_level = P.obstacle_free_level;
        }
        double *stash = nullptr;
        if constexpr (SCHED == 4) stash = A.stash + (long long)blockIdx.x * STASH_CAP * CTXD;
        if (phase == 2) {
            if (alive) b = sv.restore_context(stash + b_in * CTXD, 1);
            else b = 0;
        }
        double p0[3], v0[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            p0[c] = __ldg(A.p0 + c * A.ld + b);
            v0[c] = __ldg(A.v0 + c * A.ld + b);
            if (phase != 2) sv.goal[c] = SolverT::TRACK ? 0.0 : __ldg(A.goal + c * A.ld + b); /* not read in TRACK */
        }
        if constexpr (SolverT::TRACK) sv.set_reference(A.track_rows + b, A.ld, A.track_len, A.track_start);
        if (phase != 2) sv.has_goal = A.has_goal ? (A.has_goal[b] != 0) : true;
        if (skip_near) {
            /* a member of the priority list met in a regular round: solved (or about to be) in a
             * priority round.  The predicate of starts_near_goal on the values just loaded. */
            const double dx = sv.goal[0] - p0[0], dy = sv.goal[1] - p0[1], dz = sv.goal[2] - p0[2];
            if (sv.has_goal && dx * dx + dy * dy + dz * dz < A.prio_r2) refused = true;
        }
        const bool warm = phase != 2 && A.x_warm != nullptr && (A.warm_mask == nullptr || A.warm_mask[b] != 0);
        if (phase == 2) {
            /* nothing to start */
        } else if (warm) {
            /* plain loads: in the closed loop x_out aliases x_warm */
            const double *xw = A.x_warm + b;
            const long long ld = A.ld;
            sv.warm_start(p0, v0, [xw, ld](int row) { return xw[(long long)row * ld]; });
            if (!TILT) {
                int tilted = 0;
#pragma unroll
                for (int tt = 0; tt < TPL; ++tt)
                    tilted |= (sv.x[tt * 9 + 6] != 0.0 || sv.x[tt * 9 + 7] != 0.0) ? 1 : 0;
                if (sv.grp.any(tilted != 0) && alive && !idle_lane) { /* broken promise: no solve, say so */
                    if ((MINB < 3) && A.rows) {
                        double *row = A.rows + b * A.row_stride;
                        const int nx = (A.rows_kind == 1 ? 3 : 9) * N, nd = (A.rows_kind == 1 ? 3 : (A.rows_kind == 2 ? 9 : 19)) * N;
                        for (int i = sv.grp.lane(); i < (int)A.row_stride; i += LANES)
                            row[i] = (i == nx) ? nan("") : 0.0;
                        sv.grp.sync();
                        if (sv.grp.leader()) {
                            int *om = reinterpret_cast<int *>(row + nd + 1);
                            om[2] = 3;
                            om[4] = -2;
                        }
                    } else if (sv.grp.leader()) {
                        if (A.status) A.status[b] = 3;
                        if (A.nit) A.nit[b] = 0;
                        if (A.nfev) A.nfev[b] = 0;
                        if (A.cost) A.cost[b] = nan("");
                    }
                    refused = true;
                }
            }
        } else
            sv.cold_start(p0, v0);
        DP_TICK(0);
        SolveStats st;
        if constexpr (SCHED == 4) {
            if (phase == 1) {
                const bool run = alive && !refused;
                if (run) {
                    sv.begin();
                    if (sv.task == 0) sv.template iterate<true>();
                }
                /* unfinished problems go to the stash, packed: slot = count so far + rank among
                 * this round's continuing sub-warps */
                const int cont = (run && sv.task == 0) ? 1 : 0;
                if (sv.grp.leader()) s_cont[gib] = cont;
                __syncthreads();
                int pos = s_stash_n, total = 0;
#pragma unroll
                for (int j = 0; j < GPB; ++j) {
                    pos += (j < gib) ? s_cont[j] : 0;
                    total += s_cont[j];
                }
                if (cont) sv.save_context(stash + (long long)pos * CTXD, 1, b);
                __syncthreads();
                if (threadIdx.x == 0) s_stash_n += total;
                if (!run || cont) return;
            } else {
                for (;;) {
                    const int go = (alive && sv.task == 0) ? 1 : 0;
                    if (!__syncthreads_or(go)) break;
                    if (go) sv.template iterate<false>();
                }
                if (!alive) return;
            }
            sv.finish(st);
        } else if constexpr (LOCK) {
            /* the warps of a block start every iteration together */
            if (!refused) sv.begin();
            for (;;) {
                const int go = (!refused && sv.task == 0) ? 1 : 0;
                if (!__syncthreads_or(go)) break;
                if (go) sv.template iterate<false>();
            }
            if (refused || !alive || idle_lane) return;
            sv.finish(st);
        } else {
            if (refused) return;
            sv.minimize(st);
        }
        DP_TICK(40);
        /* outputs: `emit` writes one problem's result through per-field base pointers with
         * element stride `old` -- SoA rows of the batch (element b of every row, stride ld), or
         * the staging row in this problem's shared block (stride 1; free now, the solve is
         * over), which the group then copies out with full-line 16-byte stores.  Two inlined
         * copies, so the SoA addressing stays what it was.  (The register-capped throughput
         * builds leave the row mode out: the launcher sends row launches to the latency build,
         * whose transfers are PCIe-bound anyway.) */
        auto emit = [&](double *ox, double *ocost, double *oacc, double *oatt, double *orat, double *othr,
                        int *onit, int *onfev, int *ostat, int *otask, int *ohit, const long long old,
                        const bool check_map) {
            if (ox) {
#pragma unroll
                for (int tt = 0; tt < TPL; ++tt)
                    if (sv.act[tt]) {
#pragma unroll
                        for (int q = 0; q < 9; ++q) ox[(long long)sv.row_of(tt, q) * old] = sv.x[tt * 9 + q];
                    }
            }
            if (sv.grp.leader()) {
                if (ocost) *ocost = st.f;
                if (onit) *onit = st.nit;
                if (onfev) *onfev = st.nfev;
                if (ostat) *ostat = st.status;
                if (otask) *otask = st.task;
            }
            if (oacc || oatt || orat || othr) {
                sv.extract([=](int k, double ax, double ay, double az, double r0, double r1, double r2,
                               double w0, double w1, double w2, double th) {
                    if (oacc) {
                        oacc[(long long)(3 * k) * old] = ax;
                        oacc[(long long)(3 * k + 1) * old] = ay;
                        oacc[(long long)(3 * k + 2) * old] = az;
                    }
                    if (oatt) {
                        oatt[(long long)(3 * k) * old] = r0;
                        oatt[(long long)(3 * k + 1) * old] = r1;
                        oatt[(long long)(3 * k + 2) * old] = r2;
                    }
                    if (orat) {
                        orat[(long long)(3 * k) * old] = w0;
                        orat[(long long)(3 * k + 1) * old] = w1;
                        orat[(long long)(3 * k + 2) * old] = w2;
                    }
                    if (othr) othr[(long long)k * old] = th;
                });
            }
            if (check_map) {
                /* each lane tests its own timesteps against the map; the first colliding index is
                 * the minimum over the group (explicit_geometric_mapper.py:195-219) */
                int hit = 0x7fffffff;
#pragma unroll
                for (int tt = TPL - 1; tt >= 0; --tt)
                    if (sv.act[tt] && position_collides(A.check_grid, sv.x[tt * 9], sv.x[tt * 9 + 1], sv.x[tt * 9 + 2],
                                                        A.margin, A.threshold))
                        hit = sv.grp.lane() * TPL + tt;
                hit = sv.grp.mini(hit);
                if (sv.grp.leader()) *ohit = (hit == 0x7fffffff) ? -1 : hit;
            }
        };
        if ((MINB < 3) && A.rows != nullptr && A.rows_kind == 1) {
            /* controls row: thrust vectors, cost, counters */
            sv.grp.sync();
            for (int i = 3 * N + sv.grp.lane(); i < (int)A.row_stride; i += LANES) sm[i] = 0.0;
            sv.grp.sync();
#pragma unroll
            for (int tt = 0; tt < TPL; ++tt)
                if (sv.act[tt]) {
                    const int k = sv.grp.lane() * TPL + tt;
#pragma unroll
                    for (int c = 0; c < 3; ++c) sm[3 * k + c] = sv.x[tt * 9 + 6 + c];
                }
            if (sv.grp.leader()) {
                int *om = reinterpret_cast<int *>(sm + 3 * N + 1);
                sm[3 * N] = st.f;
                om[0] = st.nit;
                om[1] = st.nfev;
                om[2] = st.status;
                om[3] = st.task;
                om[4] = -2;
            }
            sv.grp.sync();
            double2 *dst = reinterpret_cast<double2 *>(A.rows + b * A.row_stride);
            for (int i = sv.grp.lane(); i < (int)(A.row_stride >> 1); i += LANES)
                dst[i] = make_double2(sm[2 * i], sm[2 * i + 1]);
            sv.grp.sync();
        } else if ((MINB < 3) && A.rows != nullptr) {
            /* full row (kind 0) or solution row (kind 2: x, cost, counters -- the derived arrays
             * are functions of the thrust rows of x and are left to the host) */
            sv.grp.sync();
            const bool full = (A.rows_kind == 0);
            double *oacc = sm + 9 * N + 1, *othr = oacc + 9 * N;
            int *om = reinterpret_cast<int *>(full ? othr + N : oacc);
            for (int i = (full ? 19 : 9) * N + 3 + sv.grp.lane(); i < (int)A.row_stride; i += LANES) sm[i] = 0.0;
            sv.grp.sync();
            if (!A.check_map && sv.grp.leader()) om[4] = -2; /* map check not requested */
            emit(sm, sm + 9 * N, full ? oacc : nullptr, full ? oacc + 3 * N : nullptr,
                 full ? oacc + 6 * N : nullptr, full ? othr : nullptr, om, om + 1, om + 2, om + 3, om + 4, 1,
                 A.check_map != 0);
            sv.grp.sync();
            double2 *dst = reinterpret_cast<double2 *>(A.rows + b * A.row_stride);
            for (int i = sv.grp.lane(); i < (int)(A.row_stride >> 1); i += LANES)
                dst[i] = make_double2(sm[2 * i], sm[2 * i + 1]);
            sv.grp.sync();
        } else {
            emit(A.x_out ? A.x_out + b : nullptr, A.cost ? A.cost + b : nullptr, A.acc ? A.acc + b : nullptr,
                 A.att ? A.att + b : nullptr, A.rates ? A.rates + b : nullptr,
                 A.thrust ? A.thrust + b : nullptr, A.nit ? A.nit + b : nullptr, A.nfev ? A.nfev + b : nullptr,
                 A.status ? A.status + b : nullptr, A.task ? A.task + b : nullptr,
                 A.first_hit ? A.first_hit + b : nullptr, A.ld, A.check_map != 0 && A.first_hit != nullptr);
        }
        double path[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0}; /* the plant step's p and p' - p */
        if (A.p_next && sv.grp.leader()) {
            /* reference planner model (se3_mpc_planner.py:430-431, :445-459) driven by T_0:
             * a = T_0/m - g e3;  p <- p + v dt + (0.5 a) dt^2;  v <- v + a dt.  Every operation
             * individually rounded (NumPy's order). */
            const double dt = A.plant_dt, dt2 = DP_MUL(dt, dt);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                /* the state is read again here (plain loads: p_next / v_next may alias p0 / v0)
                 * instead of being kept in 12 registers through the whole solve */
                const double pc = A.p0[c * A.ld + b], vc = A.v0[c * A.ld + b];
                const double a = DP_ADD(ddiv(sv.x[6 + c], P.mass), c == 2 ? -P.gravity : -0.0);
                const double pn = DP_ADD(DP_ADD(pc, DP_MUL(vc, dt)), DP_MUL(DP_MUL(0.5, a), dt2));
                A.p_next[c * A.ld + b] = pn;
                A.v_next[c * A.ld + b] = DP_ADD(vc, DP_MUL(a, dt));
                path[c] = pc;
                path[3 + c] = DP_ADD(pn, -pc);
            }
        }
        if (A.p_next && A.first_collision) {
            /* collision record: q_j = p + (p' - p)(j / S), j = 1..S, S = ceil(|p' - p|_inf / (res/2))
             * (at least 1, at most 64), every operation individually rounded; lanes strided over j */
#pragma unroll
            for (int c = 0; c < 6; ++c) path[c] = sv.grp.bcast(path[c], 0);
            const double h = 0.5 * A.check_grid.resolution;
            const double m = fmax(fmax(fabs(path[3]), fabs(path[4])), fabs(path[5]));
            const int S = (m <= 64.0 * h) ? max(1, (int)ceil(m / h)) : 64; /* NaN: 64 */
            bool hit = false;
            for (int j = 1 + sv.grp.lane(); j <= S && !hit; j += LANES) {
                const double t = (double)j / (double)S;
                hit = position_collides(A.check_grid, DP_ADD(path[0], DP_MUL(path[3], t)),
                                        DP_ADD(path[1], DP_MUL(path[4], t)), DP_ADD(path[2], DP_MUL(path[5], t)),
                                        A.margin, A.threshold);
            }
            hit = sv.grp.any(hit);
            if (hit && sv.grp.leader() && A.first_collision[b] == -1) A.first_collision[b] = A.step;
        }
        DP_TICK(41);
        (void)N;
    };
    if constexpr (SCHED == 1) {
        constexpr int PPW = GMap::GPW;
        const long long ntasks = (A.B + PPW - 1) / PPW;
        for (;;) {
            long long ti = 0;
            if ((threadIdx.x & 31) == 0) ti = (long long)atomicAdd(A.queue, 1ull);
            ti = __shfl_sync(0xffffffffu, ti, 0);
            if (ti >= ntasks) break;
            const long long b = ti * PPW + gib % PPW;
            if (b < A.B && !idle_lane) solve_one(b, true, 0);
            __syncwarp();
        }
    } else if constexpr (SCHED == 2) {
        __shared__ long long s_ticket;
        const long long rounds = (A.B + GPB - 1) / GPB;
        /* the list's size lives in shared memory (block-uniform, read once per round): it would
         * otherwise hold registers through the whole solve.  -1 = not read yet */
        __shared__ int s_npri;
        if (threadIdx.x == 0) s_npri = (A.prio_count == nullptr || rounds <= (long long)gridDim.x) ? 0 : -1;
        for (;;) {
            __syncthreads();
            if (threadIdx.x == 0) {
                const long long tk = (long long)atomicAdd(A.queue, 1ull);
                s_ticket = tk;
                if (tk >= (long long)gridDim.x && s_npri < 0) {
                    /* the scan kernel this launch depends on has completed: read its list.  Used
                     * when it holds a small part of the batch (a population that sits at its goals
                     * is not a set of stragglers) and fits */
#if defined(__CUDA_ARCH__)
                    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
                    const long long n = (long long)__ldcg(A.prio_count);
                    s_npri = (n > 0 && n <= PRIO_CAP && n * 64 <= A.B) ? (int)n : 0;
                }
            }
            __syncthreads();
            const long long blk = s_ticket;
            const int G = (int)gridDim.x;
            const int npri = blk >= G ? s_npri : 0;
            const int pr_rounds = (npri + GPB - 1) / GPB;
            if (blk >= rounds + pr_rounds) break;
            /* ONE call site: the solve is inlined once */
            long long b;
            bool alive;
            if (blk >= G && blk < G + pr_rounds) {
                const int i = (int)(blk - G) * GPB + gib;
#if defined(__CUDA_ARCH__)
                asm volatile("griddepcontrol.wait;" ::: "memory"); /* satisfied long ago: every reader of the list says so */
#endif
                b = (i < npri) ? (long long)__ldcg(A.prio_list + i) : 0;
                alive = i < npri && b >= (long long)G * GPB;
            } else {
                const long long br = (blk < G ? blk : blk - pr_rounds) * GPB + gib;
                b = br < A.B ? br : A.B - 1;
                alive = br < A.B;
            }
            solve_one(b, alive, 0, blk >= G + pr_rounds && npri > 0);
        }
    } else if constexpr (SCHED == 4) {
        /* Two-phase schedule.  The solves differ 3x in length (1 to 3 iterations on the bench
         * mix); run to the end side by side, a sub-warp whose problem stops after the first
         * iteration idles while its warp finishes the others.  Here a block alternates between
         *   phase 1: GPB fresh problems (one ticket) through their start and FIRST iteration --
         *            uniform work, in code specialised for "no stored pair"; the finished ones
         *            are written out, the others' contexts are stashed;
         *   phase 2: as soon as GPB contexts are stashed (or no fresh problem is left), GPB of
         *            them continue to the end, all sub-warps busy from the second iteration on. */
        __shared__ long long s_ticket;
        const long long rounds = (A.B + GPB - 1) / GPB;
        if (threadIdx.x == 0) s_stash_n = 0;
        bool fresh = true;
        for (;;) {
            __syncthreads();
            const int n = s_stash_n;
            if (n >= GPB || (!fresh && n > 0)) {
                const int take = n < GPB ? n : GPB;
                __syncthreads();
                if (threadIdx.x == 0) s_stash_n = n - take;
                solve_one((long long)(n - take + gib), gib < take, 2);
                continue;
            }
            if (!fresh) break;
            if (threadIdx.x == 0) s_ticket = (long long)atomicAdd(A.queue, 1ull);
            __syncthreads();
            const long long blk = s_ticket;
            if (blk >= rounds) {
                fresh = false;
                continue;
            }
            const long long b = blk * GPB + gib;
            solve_one(b < A.B ? b : A.B - 1, b < A.B, 1);
        }
    } else {
        /* block-uniform trip count + a warp barrier per round: the sub-warps of a warp start every
         * problem together (a sub-warp that converged early waits instead of running ahead into
         * different code) */
        const long long rounds = (A.B + GPB - 1) / GPB;
        for (long long blk = blockIdx.x; blk < rounds; blk += gridDim.x) {
            __syncwarp();
            const long long b = blk * GPB + gib;
            if constexpr (LOCK)
                solve_one(b < A.B ? b : A.B - 1, b < A.B, 0);
            else if (b < A.B && !idle_lane)
                solve_one(b, true, 0);
        }
    }
    if constexpr (SCHED == 1 || SCHED == 2 || SCHED == 4) {
        /* the last block to finish re-arms the ticket counter for the next launch that uses it */
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            if (atomicAdd(A.queue + 1, 1ull) == (unsigned long long)gridDim.x - 1ull) {
                A.queue[0] = 0ull;
                A.queue[1] = 0ull;
                if (A.prio_count) *A.prio_count = 0u;
                __threadfence();
            }
        }
    }
}

/* Solution extraction alone (se3_mpc_planner.py:582-654 for B given thrust sequences): the
 * solver's own `extract`, i.e. the code the solve kernel's epilogue runs, reachable with
 * arbitrary thrust vectors (zero-thrust steps, degenerate b1, tilted sequences) that a solve
 * only produces from special warm starts.  T: SoA rows 3k+c, row pitch ld. */
struct ExtractArgs {
    long long B, ld;
    const double *T;
    double *acc, *att, *rates, *thrust;
};

template <int LANES, int TPL, int BLOCK, bool TILT>
__global__ void __launch_bounds__(BLOCK)
se3mpc_extract_kernel(const __grid_constant__ dart_se3mpc_params P, const __grid_constant__ ExtractArgs A)
{
    using GMap = GroupMap<LANES, BLOCK>;
    constexpr int GPB = GMap::GPB;
    const int gib = GMap::gib();
    const long long rounds = (A.B + GPB - 1) / GPB;
    for (long long blk = blockIdx.x; blk < rounds; blk += gridDim.x) {
        __syncwarp();
        const long long b = blk * GPB + gib;
        if (b < A.B && !GMap::idle()) {
            Solver<typename GroupOf<LANES>::type, TPL, 0, false, TILT> sv(P, nullptr, nullptr, nullptr);
#pragma unroll
            for (int tt = 0; tt < TPL; ++tt) {
                const int k = sv.grp.lane() * TPL + tt;
#pragma unroll
                for (int q = 0; q < 9; ++q) sv.x[tt * 9 + q] = 0.0;
                if (sv.act[tt]) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) sv.x[tt * 9 + 6 + c] = A.T[(long long)(3 * k + c) * A.ld + b];
                }
            }
            const long long ld = A.ld;
            double *oacc = A.acc + b, *oatt = A.att + b, *orat = A.rates + b, *othr = A.thrust + b;
            sv.extract([=](int k, double ax, double ay, double az, double r0, double r1, double r2, double w0,
                           double w1, double w2, double th) {
                oacc[(long long)(3 * k) * ld] = ax;
                oacc[(long long)(3 * k + 1) * ld] = ay;
                oacc[(long long)(3 * k + 2) * ld] = az;
                oatt[(long long)(3 * k) * ld] = r0;
                oatt[(long long)(3 * k + 1) * ld] = r1;
                oatt[(long long)(3 * k + 2) * ld] = r2;
                orat[(long long)(3 * k) * ld] = w0;
                orat[(long long)(3 * k + 1) * ld] = w1;
                orat[(long long)(3 * k + 2) * ld] = w2;
                othr[(long long)k * ld] = th;
            });
        }
    }
}

/* the instantiations of one lane configuration: [gradient_mode][tilt], null where MODES says the
 * kernel does not exist -- tilt = 0 in the modes without a 7-slot instantiation, and the tracking
 * modes in the builds wider than their horizon limit (the 32-lane builds) */
struct KernelSet {
    const void *fn[N_MODES][2];
    const void *extract_fn[2]; /* [tilt] */
    int lanes, tpl, block, minb;
    int gpb;      /* problems per block */
    int resident; /* blocks per SM the shared-memory carve-out is sized for (default: minb) */
};

template <int LANES, int TPL, int BLK, int MINB, int GM, bool TILT>
const void *solve_fn()
{
    if constexpr ((TILT || MODES[GM].seven_slot) && (!MODES[GM].track || LANES * TPL <= MODES[GM].max_horizon))
        return (const void *)se3mpc_solve_kernel<LANES, TPL, BLK, MINB, GM, TILT>;
    else
        return nullptr;
}

template <int LANES, int TPL, int MINB, int BLK, int... GM>
KernelSet make_kernel_set(std::integer_sequence<int, GM...>)
{
    KernelSet k;
    /* tilted kernels first: in the throughput builds ptxas schedules a mode's tilted kernel
     * differently when its 7-slot twin is instantiated before it */
    ((k.fn[GM][1] = solve_fn<LANES, TPL, BLK, MINB, GM, true>()), ...);
    ((k.fn[GM][0] = solve_fn<LANES, TPL, BLK, MINB, GM, false>()), ...);
    k.extract_fn[1] = (const void *)se3mpc_extract_kernel<LANES, TPL, BLK, true>;
    k.extract_fn[0] = (const void *)se3mpc_extract_kernel<LANES, TPL, BLK, false>;
    k.lanes = LANES;
    k.tpl = TPL;
    k.block = BLK;
    k.minb = MINB;
    k.gpb = GroupMap<LANES, BLK>::GPB;
    k.resident = MINB;
    return k;
}

template <int LANES, int TPL, int MINB, int BLK>
KernelSet make_kernel_set()
{
    return make_kernel_set<LANES, TPL, MINB, BLK>(std::make_integer_sequence<int, N_MODES>());
}

/* defined one per instantiation unit */
KernelSet kernel_set_l4();
KernelSet kernel_set_l8();
KernelSet kernel_set_l16();
KernelSet kernel_set_l32();
KernelSet kernel_set_l32x2();
KernelSet kernel_set_l8_occ3();
KernelSet kernel_set_l8_b64();
KernelSet kernel_set_l16_occ3();
KernelSet kernel_set_l32_occ3();
KernelSet kernel_set_l6();
KernelSet kernel_set_l6_occ5();

} /* namespace dartb200 */
