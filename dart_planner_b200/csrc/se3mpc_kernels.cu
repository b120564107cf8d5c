/*
 * se3mpc_kernels.cu -- C ABI (include/dart_se3mpc.h) of the batched SE(3)-MPC solve: argument
 * checks, kernel choice, launch.  The kernel itself is in se3mpc_kernel.cuh / se3mpc_core.cuh;
 * its instantiations live in se3mpc_inst_*.cu.  I/O is batch-major SoA so the 32/LANES
 * problems of a warp touch consecutive addresses of every row.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>

#include "se3mpc_kernel.cuh"

using namespace dartb200;

namespace dartb200 {
__global__ void __launch_bounds__(256) se3mpc_prio_scan_kernel(const __grid_constant__ SolveArgs A)
{
    /* the solve behind this kernel may start right away: its first rounds do not need the list */
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < A.B; b += (long long)gridDim.x * blockDim.x)
        if (starts_near_goal(A, b)) {
            const unsigned slot = atomicAdd(A.prio_count, 1u);
            if (slot < (unsigned)PRIO_CAP) A.prio_list[slot] = (int)b;
        }
}
} /* namespace dartb200 */

namespace {

std::atomic<long long> g_launches{0};
thread_local char g_err[256] = "";

struct KernelChoice {
    KernelSet set; /* fn[gradient_mode][tilt]; tilt = 0: launches without warm starts, whose lateral
                    * thrust slots are exactly zero and stay zero -- 7 slots per timestep instead
                    * of 9, bit-identical results */
    int lanes, tpl, block, minb;
    int occ_blocks; /* resident blocks per SM (queried once) */
    int regs;
    unsigned long long ready; /* bit d: function attributes set on device d (they are per device) */
};

KernelChoice make_choice(const KernelSet &ks)
{
    KernelChoice k;
    k.set = ks;
    k.lanes = ks.lanes;
    k.tpl = ks.tpl;
    k.block = ks.block;
    k.minb = ks.minb;
    k.occ_blocks = 0;
    k.regs = 0;
    k.ready = 0ull;
    return k;
}

KernelChoice g_kernels[] = {
    make_choice(kernel_set_l4()), make_choice(kernel_set_l8()), make_choice(kernel_set_l16()),
    make_choice(kernel_set_l32()), make_choice(kernel_set_l32x2()),
    /* [5] the 168-register throughput build for N <= 8 (3 resident blocks per SM); [6] tuning
     * variant (64-thread blocks), DART_SE3MPC_VARIANT=<index> (tools/kbench.py) */
    make_choice(kernel_set_l8_occ3()), make_choice(kernel_set_l8_b64()),
    /* [7], [8] throughput builds for 8 < N <= 16 and 16 < N <= 32 */
    make_choice(kernel_set_l16_occ3()), make_choice(kernel_set_l32_occ3()),
    /* [9], [10] horizons 5 and 6 (the reference's class default) on 6-lane groups, five problems
     * per warp instead of four: latency build (2 blocks of 20 problems per SM) and throughput
     * build (5 blocks of 10 problems per SM).  Same results as the 8-lane builds, but measured
     * SLOWER (65 536 problems at N = 6: 275 / 268 us against 232 us in the 8-lane throughput
     * build; 1 Mi: 4.07 against 3.32 ms): the shared block caps an SM at 50 problems on 10 warps
     * against 48 on 12, five sub-warps wait for the slowest of five, and the kernel is bound by
     * latency, not by the lanes it leaves idle.  Reachable with DART_SE3MPC_VARIANT=9 / 10 only. */
    make_choice(kernel_set_l6()), make_choice(kernel_set_l6_occ5()),
};
std::mutex g_mu;
int g_sms = 0;
constexpr int QUEUE_SLOTS = 256;
unsigned long long *g_queue[64] = {nullptr};
unsigned long long g_queue_next[64] = {0};
/* context stash of the two-phase schedule: a small ring of buffers per device, one per launch in
 * flight; a launch that reuses a buffer first waits (on its stream) for the launch that used it */
constexpr int STASH_RING = 4;
struct StashBuf {
    double *ptr = nullptr;
    size_t bytes = 0;
    cudaEvent_t done = nullptr;
};
StashBuf g_stash[64][STASH_RING];
unsigned g_stash_next[64] = {0};
/* priority lists of the throughput builds ("long solves first", se3mpc_kernel.cuh): the same
 * kind of ring, one list per launch in flight: [count (16 bytes) | B problem indices] */
constexpr int PRIO_RING = 8;
constexpr long long PRIO_MIN_B = 16384; /* below this a launch is a wave or two: nothing to reorder */
StashBuf g_prio[64][PRIO_RING];
unsigned g_prio_next[64] = {0};

size_t stash_bytes_for(const KernelChoice &k, long long grid)
{
    /* upper bound of Solver::ctx_doubles(1) over the gradient modes (se3mpc_core.cuh): the
     * dynamics-consistent modes keep 6 more scalars */
    const size_t S = 9 * (size_t)k.tpl, gpb = (size_t)k.set.gpb;
    const size_t ctx = 16 + 6 + 2 * ((S + 31) / 32) + 7 + (size_t)k.lanes * (4 * S + 3 * k.tpl);
    return (size_t)grid * (2 * gpb - 1) * ctx * sizeof(double);
}

int smem_bytes(const KernelChoice &k) { return k.set.gpb * SM_DOUBLES * (int)sizeof(double); }

int set_err(cudaError_t e, const char *what)
{
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return DART_E_CUDA;
}

thread_local long long g_batch_hint = 0; /* > 0: choose the build for this many problems (the
                                          * chunks of one pipelined host batch use one build) */

std::atomic<long long> g_inflight_hint{0}; /* dart_se3mpc_set_inflight_hint: problems the caller keeps in flight */

KernelChoice *pick_kernel(int N, long long B, bool rows = false)
{
    if (g_batch_hint > B) B = g_batch_hint;
    const long long inflight = g_inflight_hint.load(std::memory_order_relaxed);
    if (inflight > B) B = inflight;
    if (rows) B = 1; /* row output exists in the latency builds only */
    int idx = N <= 4 ? 0 : N <= 8 ? 1 : N <= 16 ? 2 : N <= 32 ? 3 : 4;
    /* N <= 8: the 168-register build (3 resident blocks per SM) trades a few spills for 50 % more
     * warps in flight: +9 % at 64 Ki and 1 Mi problems, but -10 % on a single round, where
     * nothing waits for a free slot.  It takes over as soon as the latency build (2 blocks of 16
     * problems per SM) would need a second round: 6 144 problems are 43 us in one round of the
     * throughput build against 54 us in two rounds of the latency build (profiles/README.md) */
    const long long one_round = 2ll * (g_sms > 0 ? g_sms : 148) * 16; /* 2 blocks x 16 problems per SM */
    if (idx == 1 && N > 4 && B > one_round) idx = 5;
    if (idx == 2 && B >= 12288) idx = 7;
    if (idx == 3 && B >= 12288) idx = 8;
    if (const char *v = getenv("DART_SE3MPC_VARIANT")) {
        const int want = atoi(v);
        const int nk = (int)(sizeof(g_kernels) / sizeof(g_kernels[0]));
        if (want >= 0 && want < nk && g_kernels[want].lanes * g_kernels[want].tpl >= N) idx = want;
    }
    return &g_kernels[idx];
}

int prepare(KernelChoice *k)
{
    std::lock_guard<std::mutex> lk(g_mu);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        set_err(e, "cudaGetDevice");
        return DART_E_NODEVICE;
    }
    if (dev < 0 || dev >= 64) return DART_E_UNSUPPORTED;
    if (k->ready >> dev & 1ull) return DART_OK;
    if (g_sms == 0) {
        e = cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return set_err(e, "cudaDeviceGetAttribute");
    }
    const int smem = smem_bytes(*k);
    /* shared-memory share of the 256 KB L1: what `minb` resident blocks need (+1 KB each that
     * the driver reserves); the rest stays L1 for the per-lane S/Y pairs in local memory */
    int carve = (int)((long long)k->set.resident * (smem + 1024) * 100 / (228 * 1024)) + 1;
    if (carve > 100) carve = 100;
    for (const auto &by_tilt : k->set.fn)
        for (const void *fn : by_tilt) {
            if (!fn) continue; /* no such instantiation (KernelSet) */
            e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (e != cudaSuccess) return set_err(e, "cudaFuncSetAttribute(smem)");
            e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
            if (e != cudaSuccess) return set_err(e, "cudaFuncSetAttribute(carveout)");
        }
    cudaFuncAttributes fa;
    e = cudaFuncGetAttributes(&fa, k->set.fn[0][1]);
    if (e != cudaSuccess) return set_err(e, "cudaFuncGetAttributes");
    k->regs = fa.numRegs;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k->occ_blocks, k->set.fn[0][1], k->block, smem);
    if (e != cudaSuccess) return set_err(e, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
    if (k->occ_blocks < 1) k->occ_blocks = 1;
    k->ready |= 1ull << dev;
    return DART_OK;
}

/* family: the entries the caller belongs to; each family serves its own modes (ModeInfo::family) */
int check_params(const dart_se3mpc_params *p, ModeFamily family = FAM_PLAIN)
{
    if (!p || p->struct_size != (int)sizeof(dart_se3mpc_params)) return DART_E_BADARG;
    if (p->horizon < 1 || p->horizon > 64) return DART_E_UNSUPPORTED;
    if (p->max_corrections < 1 || p->max_corrections > MMAX) return DART_E_UNSUPPORTED;
    /* maxls >= 1, as SciPy requires; with 0 every solve would end ABNORMAL after one evaluation */
    if (p->max_iterations < 0 || p->max_linesearch < 1) return DART_E_BADARG;
    const ModeInfo *m = mode_info(p->gradient_mode);
    if (!m || m->family != family) return family == FAM_PLAIN ? DART_E_UNSUPPORTED : DART_E_BADARG;
    if (p->horizon > m->max_horizon) return DART_E_UNSUPPORTED;
    if (!(p->dt > 0.0) || !(p->mass > 0.0)) return DART_E_BADARG;
    if (!(p->gtol >= 0.0)) return DART_E_BADARG; /* the Cauchy step relies on it (se3mpc_core.cuh) */
    return DART_OK;
}

/* What a solve entry was called with: the modes it serves, the kind of entry, and its arguments --
 * the caller's arrays and scalars already in the launch's SolveArgs, the structs as passed.
 * check_request checks it, in the order the header documents the refusals, and completes `a`. */
enum EntryKind {
    BATCH,       /* the batch solves: optional map check into first_hit */
    ROWS,        /* dart_se3mpc_solve_batch_rows: the result and the map check in one row */
    STEP,        /* the closed-loop steps with a map or a list: optional collision record */
    STEP_NO_MAP, /* dart_se3mpc_closed_loop_step: no grid argument */
    HOST,        /* the host entries: the device solve of each chunk checks the grid */
};
struct SolveRequest {
    ModeFamily family;
    EntryKind kind;
    const dart_se3mpc_params *params;
    SolveArgs a;
    const dart_spheres *spheres = nullptr;
    const dart_track_ref *ref = nullptr;
    const dart_grid *grid = nullptr;      /* the penalty's grid; in BATCH and ROWS the map check's too */
    const dart_grid *step_grid = nullptr; /* STEP: the collision record's grid */
    int warm = 0;                         /* STEP: 0 cold, 1 warm, 2 warm with zero lateral thrust */
    SolveRequest(ModeFamily f, EntryKind k, const dart_se3mpc_params *p) : family(f), kind(k), params(p)
    {
        memset(&a, 0, sizeof(a));
    }
};

int check_spheres(const dart_spheres *s)
{
    if (!s || s->n < 0 || (s->n > 0 && !s->cxyzr)) return DART_E_BADARG;
    return DART_OK;
}

int check_request(SolveRequest &r)
{
    const dart_se3mpc_params *p = r.params;
    SolveArgs &a = r.a;
    if (r.family == FAM_SPHERES && !r.spheres) return DART_E_BADARG;
    int rc = check_params(p, r.family);
    if (rc) return rc;
    const ModeInfo &m = MODES[p->gradient_mode];
    if (r.family == FAM_TRACK) {
        const dart_track_ref *ref = r.ref;
        if (!ref || !ref->rows || ref->len < 1 || ref->start < 0) return DART_E_BADARG;
        if (m.spheres != (r.spheres != nullptr)) return DART_E_BADARG; /* mode 8 needs a list, mode 7 takes none */
        a.track_rows = ref->rows;
        a.track_len = ref->len;
        a.track_start = ref->start;
    }
    if (r.spheres) {
        if ((rc = check_spheres(r.spheres))) return rc;
        a.spheres = r.spheres->cxyzr;
        a.n_spheres = r.spheres->n;
        a.sphere_margin = r.spheres->margin;
    }
    if (a.B < 0 || a.ld < a.B || !a.p0 || !a.v0 || (!a.goal && r.family != FAM_TRACK)) return DART_E_BADARG;
    if (r.kind == HOST) return DART_OK;
    if (r.kind == ROWS) {
        if (!a.rows || a.rows_kind < 0 || a.rows_kind > 2) return DART_E_BADARG;
        if (a.rows_kind == 1 && a.check_map) return DART_E_UNSUPPORTED; /* controls rows carry no map check */
        const int need = row_stride_doubles(p->horizon, a.rows_kind);
        if (need == 0) return DART_E_UNSUPPORTED; /* the row does not fit its staging block */
        if (a.row_stride < need || (a.row_stride & 15) != 0 || a.row_stride > SM_DOUBLES ||
            ((uintptr_t)a.rows & 127) != 0)
            return DART_E_BADARG;
    }
    if (r.kind == BATCH || r.kind == ROWS) {
        if (r.kind == BATCH) a.check_map = a.first_hit != nullptr;
        if (!a.check_map && !m.grid_pen) return DART_OK;
        if (check_grid(r.grid)) return DART_E_BADARG;
        a.grid = a.check_grid = *r.grid;
        return DART_OK;
    }
    if (!a.x_out || !(a.plant_dt > 0.0)) return DART_E_BADARG;
    /* the reference window slides one sample per replan: one plant step must be one sample */
    if (r.family == FAM_TRACK && a.plant_dt != p->dt) return DART_E_BADARG;
    if (m.grid_pen && r.kind == STEP_NO_MAP) return DART_E_UNSUPPORTED;
    if (m.grid_pen && check_grid(r.grid)) return DART_E_BADARG;
    if ((r.step_grid != nullptr) != (a.first_collision != nullptr)) return DART_E_BADARG;
    if (r.step_grid && check_grid(r.step_grid)) return DART_E_BADARG;
    /* the promise of warm == 2 (zero lateral thrust) does not hold where the lateral thrust moves */
    if (m.rollout && r.warm == 2) return DART_E_BADARG;
    if (m.grid_pen) a.grid = *r.grid;
    if (r.step_grid) a.check_grid = *r.step_grid;
    a.x_warm = r.warm ? a.x_out : nullptr;
    a.no_tilt_promise = r.warm == 2;
    return DART_OK;
}

long long grid_for(const KernelChoice &k, long long B)
{
    const long long gpb = k.set.gpb;
    long long need = (B + gpb - 1) / gpb;
    long long cap = (long long)g_sms * k.occ_blocks;
    return need < cap ? need : cap;
}

} /* namespace */

extern "C" {

int dart_abi_version(void) { return DART_SE3MPC_ABI_VERSION; }
const char *dart_last_cuda_error(void) { return g_err; }
int64_t dart_launch_count(void) { return (int64_t)g_launches.load(); }

int dart_se3mpc_set_inflight_hint(int64_t problems_in_flight)
{
    if (problems_in_flight < 0) return DART_E_BADARG;
    g_inflight_hint.store(problems_in_flight, std::memory_order_relaxed);
    return DART_OK;
}
void dart_count_launch_(void) { g_launches.fetch_add(1); }

void dart_se3mpc_default_params(dart_se3mpc_params *p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->struct_size = (int)sizeof(*p);
    p->horizon = 6;             /* se3_mpc_planner.py:41 */
    p->max_iterations = 15;     /* :66 */
    p->max_corrections = 10;    /* SciPy maxcor */
    p->max_linesearch = 20;     /* SciPy maxls */
    p->max_fun = 15000;         /* SciPy maxfun */
    p->gradient_mode = 0;
    p->dt = 1.0 / 400.0;        /* timing_alignment.py:76-78 with frozen_config.py:86 */
    p->mass = 1.5;              /* :149 */
    p->gravity = 9.81;          /* :150 */
    p->pos_bound = 100.0;       /* :384 */
    p->max_velocity = 10.0;     /* :45 */
    p->max_thrust = 25.0;       /* :48 */
    p->min_thrust = 2.0;        /* :49 */
    p->tilt_thrust = 25.0 * 0.70710678118654746; /* max_thrust*sin(pi/4) (:393-397) */
    p->w_pos = 100.0;           /* :56-59 */
    p->w_vel = 10.0;
    p->w_acc = 1.0;
    p->w_thrust = 0.1;
    p->gtol = 5e-2;             /* :68, :264 */
    p->ftol = 5e-1;             /* :265 */
    p->w_obstacle = 1000.0;     /* obstacle_weight :60 (unused by the reference solve) */
    p->obstacle_free_level = 0.5; /* the mapper's prior, explicit_geometric_mapper.py:71 */
}

int dart_se3mpc_kernel_info(const dart_se3mpc_params *params, int64_t B, int32_t *lanes,
                            int32_t *block_threads, int32_t *grid_blocks, int32_t *smem,
                            int32_t *regs_per_thread)
{
    int rc = check_params(params);
    if (rc) return rc;
    KernelChoice *k = pick_kernel(params->horizon, B);
    rc = prepare(k);
    if (rc) return rc;
    if (lanes) *lanes = k->lanes;
    if (block_threads) *block_threads = k->block;
    if (grid_blocks) *grid_blocks = (int32_t)grid_for(*k, B > 0 ? B : 1);
    if (smem) *smem = smem_bytes(*k);
    if (regs_per_thread) *regs_per_thread = k->regs;
    return DART_OK;
}

static int launch_solve(const dart_se3mpc_params *params, const SolveArgs &a, void *cuda_stream)
{
    KernelChoice *k = pick_kernel(params->horizon, a.B, a.rows != nullptr);
    if (a.rows && k->minb >= 3) return DART_E_UNSUPPORTED; /* DART_SE3MPC_VARIANT forced one */
    int rc = prepare(k);
    if (rc) return rc;
    dart_se3mpc_params P = *params;
    SolveArgs args_copy = a;
    void *args[] = {(void *)&P, (void *)&args_copy};
    const long long grid_blocks = grid_for(*k, a.B);
    cudaEvent_t stash_event = nullptr, prio_event = nullptr;
    {
        /* ticket counters of the dynamic schedules: a ring of self-re-arming pairs per device, one
         * pair per launch in flight (a pair is reused 256 launches later) */
        int dev = 0;
        cudaGetDevice(&dev);
        std::lock_guard<std::mutex> lk(g_mu);
        if (!g_queue[dev]) {
            cudaError_t qe = cudaMalloc(&g_queue[dev], QUEUE_SLOTS * 2 * sizeof(unsigned long long));
            if (qe == cudaSuccess) qe = cudaMemset(g_queue[dev], 0, QUEUE_SLOTS * 2 * sizeof(unsigned long long));
            if (qe != cudaSuccess) return set_err(qe, "cudaMalloc(ticket counters)");
        }
        args_copy.queue = g_queue[dev] + 2 * (g_queue_next[dev]++ % QUEUE_SLOTS);
        /* long solves first: cold starts of a large batch in a throughput build (the predicate
         * is about cold starts; a warm-started population near its goals is not a set of stragglers).
         * Near-goal radius: where the position term of the start's objective, ~ w_pos N r^2 / 3,
         * falls below the scale of the thrust term the reference's gradient mis-states,
         * ~ w_thrust (m g)^2 N / 3 -- a scheduling heuristic, results do not depend on it.
         * Not with the fused plant step of the closed loop: that launch overwrites the state in
         * place, and a member of the list met again in a regular round is recognised by the
         * predicate on the state it loads -- after its priority-round solve has moved it, the drone
         * could leave the radius and be stepped twice (tests/test_gpu_closed_loop.py,
         * test_run_in_sub_populations_changes_no_result).  Not in the tracking modes 7 / 8: the
         * predicate reads the goal, which they do not have. */
        if (k->minb >= 3 && DART_THROUGHPUT_SCHED == 2 && a.B >= PRIO_MIN_B && a.B < (1ll << 31) &&
            a.x_warm == nullptr && a.p_next == nullptr && params->w_pos > 0.0 && a.track_rows == nullptr &&
            !getenv("DART_SE3MPC_NO_PRIO")) {
            StashBuf &pb = g_prio[dev][g_prio_next[dev]++ % PRIO_RING];
            const size_t need = 16 + (size_t)PRIO_CAP * sizeof(int); /* fixed: allocated once per slot */
            if (pb.done) {
                cudaError_t se = cudaStreamWaitEvent((cudaStream_t)cuda_stream, pb.done, 0);
                if (se != cudaSuccess) return set_err(se, "cudaStreamWaitEvent(priority list)");
            } else {
                cudaError_t se = cudaEventCreateWithFlags(&pb.done, cudaEventDisableTiming);
                if (se != cudaSuccess) return set_err(se, "cudaEventCreate(priority list)");
            }
            if (pb.bytes < need) {
                if (pb.ptr) {
                    cudaEventSynchronize(pb.done);
                    cudaFree(pb.ptr);
                }
                pb.ptr = nullptr;
                pb.bytes = 0;
                cudaError_t se = cudaMalloc(&pb.ptr, need);
                if (se == cudaSuccess) se = cudaMemsetAsync(pb.ptr, 0, 16, (cudaStream_t)cuda_stream);
                if (se != cudaSuccess) return set_err(se, "cudaMalloc(priority list)");
                pb.bytes = need;
            }
            args_copy.prio_count = reinterpret_cast<unsigned *>(pb.ptr);
            args_copy.prio_list = reinterpret_cast<int *>(reinterpret_cast<char *>(pb.ptr) + 16);
            const double hover = params->mass * params->gravity;
            args_copy.prio_r2 = params->w_thrust * hover * hover / params->w_pos * (double)params->horizon;
            prio_event = pb.done;
            long long sblocks = (a.B + 255) / 256;
            const long long cap = 8ll * (g_sms > 0 ? g_sms : 148);
            if (sblocks > cap) sblocks = cap;
            void *sargs[] = {(void *)&args_copy};
            cudaError_t se = cudaLaunchKernel((const void *)se3mpc_prio_scan_kernel, dim3((unsigned)sblocks), dim3(256),
                                              sargs, 0, (cudaStream_t)cuda_stream);
            if (se != cudaSuccess) return set_err(se, "cudaLaunchKernel(se3mpc_prio_scan)");
            g_launches.fetch_add(1);
        }
        if (k->minb >= 3 && DART_THROUGHPUT_SCHED == 4) {
            StashBuf &sb = g_stash[dev][g_stash_next[dev]++ % STASH_RING];
            const size_t need = stash_bytes_for(*k, grid_blocks);
            if (sb.done) {
                cudaError_t se = cudaStreamWaitEvent((cudaStream_t)cuda_stream, sb.done, 0);
                if (se != cudaSuccess) return set_err(se, "cudaStreamWaitEvent(stash)");
            } else {
                cudaError_t se = cudaEventCreateWithFlags(&sb.done, cudaEventDisableTiming);
                if (se != cudaSuccess) return set_err(se, "cudaEventCreate(stash)");
            }
            if (sb.bytes < need) {
                if (sb.ptr) {
                    cudaEventSynchronize(sb.done);
                    cudaFree(sb.ptr);
                }
                sb.ptr = nullptr;
                sb.bytes = 0;
                cudaError_t se = cudaMalloc(&sb.ptr, need);
                if (se != cudaSuccess) return set_err(se, "cudaMalloc(context stash)");
                sb.bytes = need;
            }
            args_copy.stash = sb.ptr;
            stash_event = sb.done;
        }
    }
    int gm = params->gradient_mode;
    const int cold = ((a.x_warm == nullptr || a.no_tilt_promise) && MODES[gm].seven_slot &&
                      !getenv("DART_SE3MPC_NO_COLD")) ? 0 : 1;
    /* an empty sphere list runs the plain mode's own kernel (mode 5 -> 0, 6 -> 3, 8 -> 7): the same
     * results bit for bit, which a separate kernel cannot promise -- ptxas contracts the plain
     * products and sums of the shared solver code kernel by kernel (DESIGN.md 5e) */
    if (MODES[gm].spheres && a.n_spheres == 0) gm = MODES[gm].empty_spheres;
    const void *fn = k->set.fn[gm][cold];
    if (!fn) return DART_E_UNSUPPORTED; /* modes 7 / 8 forced onto a 32-lane build (DART_SE3MPC_VARIANT) */
    cudaError_t e;
    if (prio_event) {
        /* programmatic dependent launch: the solve may begin while the scan in front of it runs */
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3((unsigned)grid_blocks);
        cfg.blockDim = dim3(k->block);
        cfg.dynamicSmemBytes = smem_bytes(*k);
        cfg.stream = (cudaStream_t)cuda_stream;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr.val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = &attr;
        cfg.numAttrs = 1;
        e = cudaLaunchKernelExC(&cfg, fn, args);
    } else
        e = cudaLaunchKernel(fn, dim3((unsigned)grid_blocks), dim3(k->block), args, smem_bytes(*k),
                             (cudaStream_t)cuda_stream);
    if (e != cudaSuccess) return set_err(e, "cudaLaunchKernel(se3mpc_solve)");
    if (stash_event) cudaEventRecord(stash_event, (cudaStream_t)cuda_stream);
    if (prio_event) cudaEventRecord(prio_event, (cudaStream_t)cuda_stream);
    g_launches.fetch_add(1);
    return DART_OK;
}

/* a checked request runs on the device; B == 0 ends after the checks */
static int solve(SolveRequest &r, void *cuda_stream)
{
    const int rc = check_request(r);
    if (rc || r.a.B == 0) return rc;
    return launch_solve(r.params, r.a, cuda_stream);
}

/* the arguments every batch solve shares */
static SolveArgs &batch_args(SolveRequest &r, int64_t B, int64_t ld, const double *p0, const double *v0,
                             const double *goal, const uint8_t *has_goal, const double *x_warm,
                             const uint8_t *warm_mask)
{
    SolveArgs &a = r.a;
    a.B = B; a.ld = ld;
    a.p0 = p0; a.v0 = v0; a.goal = goal; a.has_goal = has_goal;
    a.x_warm = x_warm; a.warm_mask = warm_mask;
    return a;
}

static void set_outputs(SolveArgs &a, double *x_out, double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                        int32_t *task, double *acc, double *att, double *rates, double *thrust)
{
    a.x_out = x_out; a.cost = cost; a.nit = nit; a.nfev = nfev; a.status = status; a.task = task;
    a.acc = acc; a.att = att; a.rates = rates; a.thrust = thrust;
}

/* the arguments every closed-loop step shares: the state p / v is stepped in place, x is the warm
 * start (warm != 0) and the new plan */
static SolveArgs &step_args(SolveRequest &r, int64_t B, int64_t ld, double *p, double *v, const double *goal,
                            const uint8_t *has_goal, double *x, int32_t warm, double *cost, int32_t *nit,
                            int32_t *nfev, int32_t *status, double plant_dt)
{
    SolveArgs &a = r.a;
    a.B = B; a.ld = ld;
    a.p0 = a.p_next = p; a.v0 = a.v_next = v; a.goal = goal; a.has_goal = has_goal;
    a.x_out = x; a.cost = cost; a.nit = nit; a.nfev = nfev; a.status = status;
    a.plant_dt = plant_dt;
    r.warm = warm;
    return a;
}

int dart_se3mpc_solve_batch_map(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                const double *p0, const double *v0, const double *goal,
                                const uint8_t *has_goal, const double *x_warm,
                                const uint8_t *warm_mask, double *x_out, double *cost, int32_t *nit,
                                int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                double *att, double *rates, double *thrust, const dart_grid *grid,
                                double margin, double threshold, int32_t *first_hit,
                                void *cuda_stream)
{
    SolveRequest r(FAM_PLAIN, BATCH, params);
    SolveArgs &a = batch_args(r, B, ld, p0, v0, goal, has_goal, x_warm, warm_mask);
    set_outputs(a, x_out, cost, nit, nfev, status, task, acc, att, rates, thrust);
    r.grid = grid; a.margin = margin; a.threshold = threshold; a.first_hit = first_hit;
    return solve(r, cuda_stream);
}

int dart_se3mpc_solve_batch_spheres(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                    const double *p0, const double *v0, const double *goal,
                                    const uint8_t *has_goal, const double *x_warm,
                                    const uint8_t *warm_mask, double *x_out, double *cost, int32_t *nit,
                                    int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                    double *att, double *rates, double *thrust, const dart_spheres *spheres,
                                    const dart_grid *grid, double margin, double threshold,
                                    int32_t *first_hit, void *cuda_stream)
{
    SolveRequest r(FAM_SPHERES, BATCH, params);
    SolveArgs &a = batch_args(r, B, ld, p0, v0, goal, has_goal, x_warm, warm_mask);
    set_outputs(a, x_out, cost, nit, nfev, status, task, acc, att, rates, thrust);
    r.spheres = spheres;
    r.grid = grid; a.margin = margin; a.threshold = threshold; a.first_hit = first_hit;
    return solve(r, cuda_stream);
}

int dart_se3mpc_solve_batch_track(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                  const double *p0, const double *v0, const uint8_t *has_goal,
                                  const double *x_warm, const uint8_t *warm_mask, double *x_out, double *cost,
                                  int32_t *nit, int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                  double *att, double *rates, double *thrust, const dart_track_ref *ref,
                                  const dart_spheres *spheres, const dart_grid *grid, double margin,
                                  double threshold, int32_t *first_hit, void *cuda_stream)
{
    SolveRequest r(FAM_TRACK, BATCH, params);
    SolveArgs &a = batch_args(r, B, ld, p0, v0, nullptr, has_goal, x_warm, warm_mask);
    set_outputs(a, x_out, cost, nit, nfev, status, task, acc, att, rates, thrust);
    r.ref = ref;
    r.spheres = spheres;
    r.grid = grid; a.margin = margin; a.threshold = threshold; a.first_hit = first_hit;
    return solve(r, cuda_stream);
}

int dart_se3mpc_solve_batch(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                            const double *p0, const double *v0, const double *goal,
                            const uint8_t *has_goal, const double *x_warm,
                            const uint8_t *warm_mask, double *x_out, double *cost, int32_t *nit,
                            int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                            double *att, double *rates, double *thrust, void *cuda_stream)
{
    return dart_se3mpc_solve_batch_map(params, B, ld, p0, v0, goal, has_goal, x_warm, warm_mask, x_out,
                                       cost, nit, nfev, status, task, acc, att, rates, thrust, nullptr,
                                       0.0, 0.0, nullptr, cuda_stream);
}

int dart_se3mpc_solve_batch_rows(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                 const double *p0, const double *v0, const double *goal,
                                 const uint8_t *has_goal, const double *x_warm,
                                 const uint8_t *warm_mask, double *rows, int64_t row_stride,
                                 int32_t row_kind, const dart_grid *grid, double margin,
                                 double threshold, int32_t check_map, void *cuda_stream)
{
    SolveRequest r(FAM_PLAIN, ROWS, params);
    SolveArgs &a = batch_args(r, B, ld, p0, v0, goal, has_goal, x_warm, warm_mask);
    a.rows = rows; a.row_stride = row_stride; a.rows_kind = row_kind;
    r.grid = grid; a.margin = margin; a.threshold = threshold; a.check_map = check_map != 0;
    return solve(r, cuda_stream);
}

int dart_se3mpc_closed_loop_step(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                 double *v, const double *goal, const uint8_t *has_goal, double *x,
                                 int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                 int32_t *status, double plant_dt, void *cuda_stream)
{
    SolveRequest r(FAM_PLAIN, STEP_NO_MAP, params);
    step_args(r, B, ld, p, v, goal, has_goal, x, warm, cost, nit, nfev, status, plant_dt);
    return solve(r, cuda_stream);
}

int dart_se3mpc_closed_loop_step_map(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                     double *v, const double *goal, const uint8_t *has_goal, double *x,
                                     int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                     int32_t *status, double plant_dt, const dart_grid *penalty_grid,
                                     const dart_grid *check_grid, double margin, double threshold,
                                     int32_t step, int32_t *first_collision, void *cuda_stream)
{
    SolveRequest r(FAM_PLAIN, STEP, params);
    SolveArgs &a = step_args(r, B, ld, p, v, goal, has_goal, x, warm, cost, nit, nfev, status, plant_dt);
    r.grid = penalty_grid;
    r.step_grid = check_grid; a.margin = margin; a.threshold = threshold; a.step = step;
    a.first_collision = first_collision;
    return solve(r, cuda_stream);
}

int dart_se3mpc_closed_loop_step_spheres(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                         double *v, const double *goal, const uint8_t *has_goal, double *x,
                                         int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                         int32_t *status, double plant_dt, const dart_spheres *spheres,
                                         const dart_grid *check_grid, double margin, double threshold,
                                         int32_t step, int32_t *first_collision, void *cuda_stream)
{
    SolveRequest r(FAM_SPHERES, STEP, params);
    SolveArgs &a = step_args(r, B, ld, p, v, goal, has_goal, x, warm, cost, nit, nfev, status, plant_dt);
    r.spheres = spheres;
    r.step_grid = check_grid; a.margin = margin; a.threshold = threshold; a.step = step;
    a.first_collision = first_collision;
    return solve(r, cuda_stream);
}

int dart_se3mpc_closed_loop_step_track(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                       double *v, const uint8_t *has_goal, double *x, int32_t warm, double *cost,
                                       int32_t *nit, int32_t *nfev, int32_t *status, double plant_dt,
                                       const dart_track_ref *ref, const dart_spheres *spheres,
                                       const dart_grid *check_grid, double margin, double threshold,
                                       int32_t step, int32_t *first_collision, void *cuda_stream)
{
    SolveRequest r(FAM_TRACK, STEP, params);
    SolveArgs &a = step_args(r, B, ld, p, v, nullptr, has_goal, x, warm, cost, nit, nfev, status, plant_dt);
    r.ref = ref;
    r.spheres = spheres;
    r.step_grid = check_grid; a.margin = margin; a.threshold = threshold; a.step = step;
    a.first_collision = first_collision;
    return solve(r, cuda_stream);
}

int dart_se3mpc_extract_batch(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                              const double *thrust_vectors, double *acc, double *att, double *rates,
                              double *thrust, int32_t untilted, void *cuda_stream)
{
    int rc = check_params(params);
    if (rc) return rc;
    if (B < 0 || ld < B || !thrust_vectors || !acc || !att || !rates || !thrust) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    KernelChoice *k = pick_kernel(params->horizon, 1);
    rc = prepare(k);
    if (rc) return rc;
    dart_se3mpc_params P = *params;
    ExtractArgs a;
    a.B = B; a.ld = ld; a.T = thrust_vectors;
    a.acc = acc; a.att = att; a.rates = rates; a.thrust = thrust;
    void *args[] = {(void *)&P, (void *)&a};
    const long long gpb = k->set.gpb;
    long long grid = (B + gpb - 1) / gpb;
    const long long cap = (long long)g_sms * 8;
    if (grid > cap) grid = cap;
    cudaError_t e = cudaLaunchKernel(k->set.extract_fn[untilted ? 0 : 1], dim3((unsigned)grid), dim3(k->block),
                                     args, 0, (cudaStream_t)cuda_stream);
    if (e != cudaSuccess) return set_err(e, "cudaLaunchKernel(se3mpc_extract)");
    g_launches.fetch_add(1);
    return DART_OK;
}

int64_t dart_se3mpc_row_stride(const dart_se3mpc_params *params, int32_t row_kind)
{
    if (check_params(params) || row_kind < 0 || row_kind > 2) return 0;
    return (int64_t)row_stride_doubles(params->horizon, row_kind);
}

/* ---- host-buffer entry: staged through a cached per-thread device workspace --------------- */
namespace {
struct HostWs {
    void *dev = nullptr;
    size_t cap = 0;
    void *pin = nullptr; /* pinned host mirror of the workspace (small batches) */
    size_t pin_cap = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr; /* second lane of the chunk pipeline (large batches) */
    cudaEvent_t spheres_up = nullptr; /* the sphere list's upload, awaited by the second lane */
    int device = -1;                /* the device everything above belongs to */
};
thread_local HostWs g_ws;

/* one block of rows of the workspace: the caller's array of `rows` rows of B elements of esz bytes
 * (NULL: not passed, not copied) and its place in the workspace, rows of Bp elements from byte `off` */
struct WsRows {
    const void *user;
    size_t off, rows, esz;
};

/* the host's cudaMemcpy2D: `rows` rows of `width` bytes */
void copy_rows(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width, size_t rows)
{
    for (size_t r = 0; r < rows; ++r) memcpy((char *)dst + r * dpitch, (const char *)src + r * spitch, width);
}
}

void dart_se3mpc_release_thread_workspace(void)
{
    if (g_ws.device >= 0) {
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(g_ws.device);
        if (g_ws.stream) cudaStreamSynchronize(g_ws.stream);
        if (g_ws.stream2) cudaStreamSynchronize(g_ws.stream2);
        if (g_ws.dev) cudaFree(g_ws.dev);
        if (g_ws.stream) cudaStreamDestroy(g_ws.stream);
        if (g_ws.stream2) cudaStreamDestroy(g_ws.stream2);
        if (g_ws.spheres_up) cudaEventDestroy(g_ws.spheres_up);
        cudaSetDevice(cur);
    }
    if (g_ws.pin) cudaFreeHost(g_ws.pin);
    g_ws = HostWs();
}

/* the host entries: r holds the caller's host arrays; the sphere list, if any, is staged behind the
 * workspace */
static int solve_host(SolveRequest &r)
{
    int rc = check_request(r);
    if (rc) return rc;
    const SolveArgs &u = r.a;
    const int64_t B = u.B;
    if (B == 0) return DART_OK;
    const size_t N = (size_t)r.params->horizon;
    const dart_spheres *spheres = r.spheres;
    /* small batches (the drop-in planner's single solve): no copies at all -- the kernel reads its
     * inputs from and writes its results to a mapped pinned block over PCIe (zero-copy: one
     * launch and one synchronise; 62 us instead of 85 us at 512 problems); large batches copy
     * rows straight from / to the caller's buffers */
    const bool staged = B <= 512;
    const size_t Bp = staged ? (size_t)((B + 3) / 4 * 4) : (size_t)((B + 31) / 32 * 32);
    /* workspace layout for row pitch Bp (elements): fp64 rows [p0 3 | v0 3 | goal 3 | x_warm 9N |
     * x 9N | cost 1 | acc 3N | att 3N | rates 3N | thrust N], int32 rows [nit nfev status task],
     * u8 row [has_goal] */
    const size_t d8 = Bp * 8, x_off = (9 + 9 * N) * d8, acc_off = x_off + (9 * N + 1) * d8;
    const size_t int_off = acc_off + 10 * N * d8, hg_off = int_off + 4 * Bp * 4;
    const WsRows in[] = {{u.p0, 0, 3, 8}, {u.v0, 3 * d8, 3, 8}, {u.goal, 6 * d8, 3, 8},
                         {u.has_goal, hg_off, 1, 1}, {u.x_warm, 9 * d8, 9 * N, 8}};
    const WsRows out[] = {{u.x_out, x_off, 9 * N, 8},           {u.cost, x_off + 9 * N * d8, 1, 8},
                          {u.nit, int_off, 1, 4},               {u.nfev, int_off + 4 * Bp, 1, 4},
                          {u.status, int_off + 8 * Bp, 1, 4},   {u.acc, acc_off, 3 * N, 8},
                          {u.att, acc_off + 3 * N * d8, 3 * N, 8}, {u.rates, acc_off + 6 * N * d8, 3 * N, 8},
                          {u.thrust, acc_off + 9 * N * d8, N, 8}};
    /* the sphere list, if any, follows the workspace: [n][4] doubles at a 16-byte offset */
    const size_t sph_off = (hg_off + (Bp + 7) / 8 * 8 + 15) / 16 * 16;
    const size_t sph_bytes = spheres ? (size_t)spheres->n * 4 * sizeof(double) : 0;
    const size_t ws_bytes = sph_off + sph_bytes;
    cudaError_t e;
    {
        int dev = 0;
        e = cudaGetDevice(&dev);
        if (e != cudaSuccess) {
            set_err(e, "cudaGetDevice");
            return DART_E_NODEVICE;
        }
        if (g_ws.device != dev) { /* the calling thread moved to another GPU: start over there */
            if (g_ws.device >= 0) {
                cudaSetDevice(g_ws.device);
                if (g_ws.dev) cudaFree(g_ws.dev);
                if (g_ws.stream) cudaStreamDestroy(g_ws.stream);
                if (g_ws.stream2) cudaStreamDestroy(g_ws.stream2);
                if (g_ws.spheres_up) cudaEventDestroy(g_ws.spheres_up);
                cudaSetDevice(dev);
            }
            g_ws.dev = nullptr;
            g_ws.cap = 0;
            g_ws.stream = g_ws.stream2 = nullptr;
            g_ws.spheres_up = nullptr;
            g_ws.device = dev;
        }
    }
    if (!g_ws.stream) {
        e = cudaStreamCreateWithFlags(&g_ws.stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) return set_err(e, "cudaStreamCreate");
    }
    if (!staged && g_ws.cap < ws_bytes) {
        if (g_ws.dev) cudaFree(g_ws.dev);
        g_ws.dev = nullptr;
        g_ws.cap = 0;
        e = cudaMalloc(&g_ws.dev, ws_bytes);
        if (e != cudaSuccess) return set_err(e, "cudaMalloc(workspace)");
        g_ws.cap = ws_bytes;
    }
    if (staged && g_ws.pin_cap < ws_bytes) {
        if (g_ws.pin) cudaFreeHost(g_ws.pin);
        g_ws.pin = nullptr;
        g_ws.pin_cap = 0;
        e = cudaHostAlloc(&g_ws.pin, ws_bytes, cudaHostAllocMapped | cudaHostAllocPortable);
        if (e != cudaSuccess) return set_err(e, "cudaHostAlloc(staging)");
        g_ws.pin_cap = ws_bytes;
    }
    cudaStream_t s = g_ws.stream;
    char *base = (char *)g_ws.dev;
    if (staged) { /* the kernel's view of the pinned block */
        void *mapped = nullptr;
        e = cudaHostGetDevicePointer(&mapped, g_ws.pin, 0);
        if (e != cudaSuccess) return set_err(e, "cudaHostGetDevicePointer");
        base = (char *)mapped;
    }
    /* the device copy of the list the solves read (uploaded once per call) */
    dart_spheres dsph;
    if (spheres) {
        dsph = *spheres;
        dsph.cxyzr = sph_bytes ? (const double *)(base + sph_off) : nullptr;
        if (sph_bytes && staged)
            memcpy((char *)g_ws.pin + sph_off, spheres->cxyzr, sph_bytes);
        else if (sph_bytes) {
            e = cudaMemcpyAsync(base + sph_off, spheres->cxyzr, sph_bytes, cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) return set_err(e, "cudaMemcpyAsync H2D (spheres)");
        }
    }
    /* the device solve of problems [c0, c0 + cb) on the workspace's rows; only the outputs the
     * caller asked for are computed and written */
    auto run = [&](int64_t c0, int64_t cb, cudaStream_t cs) {
        auto at = [&](const WsRows &w) { return w.user ? base + w.off + c0 * w.esz : nullptr; };
        SolveRequest d(r.family, BATCH, r.params);
        d.spheres = spheres ? &dsph : nullptr;
        SolveArgs &a = batch_args(d, cb, (int64_t)Bp, (const double *)at(in[0]), (const double *)at(in[1]),
                                  (const double *)at(in[2]), (const uint8_t *)at(in[3]), (const double *)at(in[4]),
                                  nullptr);
        set_outputs(a, (double *)at(out[0]), (double *)at(out[1]), (int32_t *)at(out[2]), (int32_t *)at(out[3]),
                    (int32_t *)at(out[4]), nullptr, (double *)at(out[5]), (double *)at(out[6]),
                    (double *)at(out[7]), (double *)at(out[8]));
        return solve(d, (void *)cs);
    };
    if (staged) {
        char *h = (char *)g_ws.pin;
        for (const WsRows &w : in)
            if (w.user) copy_rows(h + w.off, Bp * w.esz, w.user, (size_t)B * w.esz, (size_t)B * w.esz, w.rows);
        rc = run(0, B, s);
        if (rc) return rc;
        e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return set_err(e, "cudaStreamSynchronize");
        for (const WsRows &w : out)
            if (w.user)
                copy_rows(const_cast<void *>(w.user), (size_t)B * w.esz, h + w.off, Bp * w.esz, (size_t)B * w.esz,
                          w.rows);
        return DART_OK;
    }
    /* Large batch: chunks of 32768 problems alternate between two streams, each doing its own
     * pitched H2D rows -> solve -> pitched D2H rows, so the read-back of chunk i (the dominant
     * cost: 1.3 KB per solve over PCIe) overlaps the solve of chunk i+1 and the upload of chunk
     * i+2.  Fully asynchronous when the caller's buffers are pinned.  Below 65536 problems: one
     * chunk on one stream. */
    const bool pipelined = B >= 65536;
    const int64_t chunk = pipelined ? 32768 : B;
    if (pipelined) {
        if (!g_ws.stream2) {
            e = cudaStreamCreateWithFlags(&g_ws.stream2, cudaStreamNonBlocking);
            if (e != cudaSuccess) return set_err(e, "cudaStreamCreate");
        }
        if (sph_bytes) { /* the list was uploaded on the first lane: the second waits for it */
            if (!g_ws.spheres_up) {
                e = cudaEventCreateWithFlags(&g_ws.spheres_up, cudaEventDisableTiming);
                if (e != cudaSuccess) return set_err(e, "cudaEventCreate(spheres)");
            }
            e = cudaEventRecord(g_ws.spheres_up, g_ws.stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(g_ws.stream2, g_ws.spheres_up, 0);
            if (e != cudaSuccess) return set_err(e, "cudaStreamWaitEvent(spheres)");
        }
    }
    /* on a failure mid-loop the copies already queued still write into the caller's buffers:
     * wait for them before handing the buffers back */
    auto drain = [&]() {
        if (!pipelined) return;
        cudaStreamSynchronize(g_ws.stream);
        cudaStreamSynchronize(g_ws.stream2);
    };
    struct HintScope { /* every chunk runs the build chosen for the whole batch */
        explicit HintScope(long long b) { g_batch_hint = b; }
        ~HintScope() { g_batch_hint = 0; }
    } hint_scope(B);
    int ci = 0;
    for (int64_t c0 = 0; c0 < B; c0 += chunk, ++ci) {
        const int64_t cb = (B - c0 < chunk) ? (B - c0) : chunk;
        cudaStream_t cs = (ci & 1) ? g_ws.stream2 : g_ws.stream;
        for (const WsRows &w : in) {
            if (!w.user) continue;
            e = cudaMemcpy2DAsync(base + w.off + c0 * w.esz, Bp * w.esz, (const char *)w.user + c0 * w.esz,
                                  (size_t)B * w.esz, (size_t)cb * w.esz, w.rows, cudaMemcpyHostToDevice, cs);
            if (e != cudaSuccess) return drain(), set_err(e, "cudaMemcpy2DAsync H2D");
        }
        rc = run(c0, cb, cs);
        if (rc) return drain(), rc;
        for (const WsRows &w : out) {
            if (!w.user) continue;
            e = cudaMemcpy2DAsync((char *)const_cast<void *>(w.user) + c0 * w.esz, (size_t)B * w.esz,
                                  base + w.off + c0 * w.esz, Bp * w.esz, (size_t)cb * w.esz, w.rows,
                                  cudaMemcpyDeviceToHost, cs);
            if (e != cudaSuccess) return drain(), set_err(e, "cudaMemcpy2DAsync D2H");
        }
    }
    e = cudaStreamSynchronize(g_ws.stream);
    if (e == cudaSuccess && pipelined) e = cudaStreamSynchronize(g_ws.stream2);
    if (e != cudaSuccess) return set_err(e, "cudaStreamSynchronize");
    return DART_OK;
}

int dart_se3mpc_solve_batch_host(const dart_se3mpc_params *params, int64_t B,
                                 const double *p0, const double *v0, const double *goal,
                                 const uint8_t *has_goal, const double *x_warm, double *x_out,
                                 double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                                 double *acc, double *att, double *rates, double *thrust)
{
    SolveRequest r(FAM_PLAIN, HOST, params);
    SolveArgs &a = batch_args(r, B, B, p0, v0, goal, has_goal, x_warm, nullptr);
    set_outputs(a, x_out, cost, nit, nfev, status, nullptr, acc, att, rates, thrust);
    return solve_host(r);
}

int dart_se3mpc_solve_batch_host_spheres(const dart_se3mpc_params *params, int64_t B,
                                         const double *p0, const double *v0, const double *goal,
                                         const uint8_t *has_goal, const double *x_warm, double *x_out,
                                         double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                                         double *acc, double *att, double *rates, double *thrust,
                                         const dart_spheres *spheres)
{
    SolveRequest r(FAM_SPHERES, HOST, params);
    SolveArgs &a = batch_args(r, B, B, p0, v0, goal, has_goal, x_warm, nullptr);
    set_outputs(a, x_out, cost, nit, nfev, status, nullptr, acc, att, rates, thrust);
    r.spheres = spheres;
    return solve_host(r);
}

} /* extern "C" */
