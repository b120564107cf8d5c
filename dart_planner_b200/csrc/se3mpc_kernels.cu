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
    const void *fns[] = {k->set.fn[0][0], k->set.fn[0][1], k->set.fn[1][0], k->set.fn[1][1],
                         k->set.fn[2][0], k->set.fn[2][1], k->set.fn[3][1], k->set.fn[4][1],
                         k->set.fn[5][0], k->set.fn[5][1], k->set.fn[6][1], k->set.fn[7][1],
                         k->set.fn[8][1]};
    for (const void *fn : fns) {
        if (!fn) continue; /* modes 7 / 8 in the 32-lane builds */
        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return set_err(e, "cudaFuncSetAttribute(smem)");
    }
    /* shared-memory share of the 256 KB L1: what `minb` resident blocks need (+1 KB each that
     * the driver reserves); the rest stays L1 for the per-lane S/Y pairs in local memory */
    int carve = (int)((long long)k->set.resident * (smem + 1024) * 100 / (228 * 1024)) + 1;
    if (carve > 100) carve = 100;
    for (const void *fn : fns) {
        if (!fn) continue;
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

/* the dynamics-consistent modes: thrusts are the only variables, P / V their rollout */
bool rollout_mode(int gm) { return gm == 3 || gm == 4 || gm == 6 || gm == 7 || gm == 8; }

/* spheres: the caller is one of the _spheres entries, which serve modes 5 and 6 only; track: one of
 * the _track entries, which serve modes 7 and 8 only; every other entry serves modes 0..4 */
int check_params(const dart_se3mpc_params *p, bool spheres = false, bool track = false)
{
    if (!p || p->struct_size != (int)sizeof(dart_se3mpc_params)) return DART_E_BADARG;
    if (p->horizon < 1 || p->horizon > 64) return DART_E_UNSUPPORTED;
    if (p->max_corrections < 1 || p->max_corrections > MMAX) return DART_E_UNSUPPORTED;
    /* maxls >= 1, as SciPy requires; with 0 every solve would end ABNORMAL after one evaluation */
    if (p->max_iterations < 0 || p->max_linesearch < 1) return DART_E_BADARG;
    if (track) {
        if (p->gradient_mode != 7 && p->gradient_mode != 8) return DART_E_BADARG;
    } else if (spheres) {
        if (p->gradient_mode != 5 && p->gradient_mode != 6) return DART_E_BADARG;
    } else if (p->gradient_mode < 0 || p->gradient_mode > 4)
        return DART_E_UNSUPPORTED;
    /* dynamics-consistent modes: verified against the oracle up to the 16-lane builds; on 32-lane
     * groups (horizons 17..64) the scan's rounding makes 5-7 % of the solves take other iteration
     * counts than the sequential oracle at tolerance 1e-3 (DESIGN.md 5c) */
    if (rollout_mode(p->gradient_mode) && p->horizon > 16) return DART_E_UNSUPPORTED;
    if (!(p->dt > 0.0) || !(p->mass > 0.0)) return DART_E_BADARG;
    if (!(p->gtol >= 0.0)) return DART_E_BADARG; /* the Cauchy step relies on it (se3mpc_core.cuh) */
    return DART_OK;
}

int check_spheres(const dart_spheres *s)
{
    if (!s || s->n < 0 || (s->n > 0 && !s->cxyzr)) return DART_E_BADARG;
    return DART_OK;
}

void set_spheres(SolveArgs &a, const dart_spheres *s)
{
    if (!s) return;
    a.spheres = s->cxyzr;
    a.n_spheres = s->n;
    a.sphere_margin = s->margin;
}

/* the reference and sphere list of a _track entry (mode 7 takes no spheres, mode 8 needs them) */
int check_track(const dart_se3mpc_params *p, const dart_track_ref *ref, const dart_spheres *s)
{
    if (!ref || !ref->rows || ref->len < 1 || ref->start < 0) return DART_E_BADARG;
    if ((p->gradient_mode == 8) != (s != nullptr)) return DART_E_BADARG;
    return s ? check_spheres(s) : DART_OK;
}

void set_track(SolveArgs &a, const dart_track_ref *ref)
{
    if (!ref) return;
    a.track_rows = ref->rows;
    a.track_len = ref->len;
    a.track_start = ref->start;
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
    /* never the 7-slot instantiation in the dynamics-consistent modes: their lateral thrust moves */
    const int cold = ((a.x_warm == nullptr || a.no_tilt_promise) && !rollout_mode(params->gradient_mode) &&
                      !getenv("DART_SE3MPC_NO_COLD")) ? 0 : 1;
    /* an empty sphere list runs the plain mode's own kernel (mode 5 -> 0, 6 -> 3): the same results
     * bit for bit, which a separate kernel cannot promise -- ptxas contracts the plain products and
     * sums of the shared solver code kernel by kernel (DESIGN.md 5e) */
    int gm = params->gradient_mode;
    if ((gm == 5 || gm == 6 || gm == 8) && a.n_spheres == 0) gm = (gm == 5) ? 0 : (gm == 6 ? 3 : 7);
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

/* the device solve of dart_se3mpc_solve_batch_map (spheres == NULL) and
 * dart_se3mpc_solve_batch_spheres */
static int solve_batch_impl(const dart_se3mpc_params *params, int64_t B, int64_t ld, const double *p0,
                            const double *v0, const double *goal, const uint8_t *has_goal,
                            const double *x_warm, const uint8_t *warm_mask, double *x_out, double *cost,
                            int32_t *nit, int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                            double *att, double *rates, double *thrust, const dart_grid *grid, double margin,
                            double threshold, int32_t *first_hit, const dart_spheres *spheres,
                            void *cuda_stream, const dart_track_ref *ref = nullptr, bool track = false)
{
    int rc = check_params(params, spheres != nullptr, track);
    if (rc) return rc;
    if (track && (rc = check_track(params, ref, spheres))) return rc;
    if (!track && spheres && (rc = check_spheres(spheres))) return rc;
    if (B < 0 || ld < B || !p0 || !v0 || (!goal && !track)) return DART_E_BADARG;
    const bool need_grid = first_hit != nullptr || params->gradient_mode == 2 || params->gradient_mode == 4;
    if (need_grid && (!grid || !grid->occ || grid->nx <= 0 || grid->ny <= 0 || grid->nz <= 0 ||
                      !(grid->resolution > 0.0)))
        return DART_E_BADARG;
    if (B == 0) return DART_OK;
    SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.ld = ld;
    a.p0 = p0; a.v0 = v0; a.goal = goal; a.has_goal = has_goal;
    a.x_warm = x_warm; a.warm_mask = warm_mask;
    a.x_out = x_out; a.cost = cost; a.nit = nit; a.nfev = nfev; a.status = status; a.task = task;
    a.acc = acc; a.att = att; a.rates = rates; a.thrust = thrust;
    if (need_grid) a.grid = a.check_grid = *grid;
    if (first_hit) {
        a.margin = margin;
        a.threshold = threshold;
        a.first_hit = first_hit;
        a.check_map = 1;
    }
    set_spheres(a, spheres);
    set_track(a, ref);
    return launch_solve(params, a, cuda_stream);
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
    return solve_batch_impl(params, B, ld, p0, v0, goal, has_goal, x_warm, warm_mask, x_out, cost, nit, nfev,
                            status, task, acc, att, rates, thrust, grid, margin, threshold, first_hit, nullptr,
                            cuda_stream);
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
    if (!spheres) return DART_E_BADARG;
    return solve_batch_impl(params, B, ld, p0, v0, goal, has_goal, x_warm, warm_mask, x_out, cost, nit, nfev,
                            status, task, acc, att, rates, thrust, grid, margin, threshold, first_hit, spheres,
                            cuda_stream);
}

int dart_se3mpc_closed_loop_step(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                 double *v, const double *goal, const uint8_t *has_goal, double *x,
                                 int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                 int32_t *status, double plant_dt, void *cuda_stream)
{
    int rc = check_params(params);
    if (rc) return rc;
    if (B < 0 || ld < B || !p || !v || !goal || !x || !(plant_dt > 0.0)) return DART_E_BADARG;
    /* no map argument here: no obstacle penalty */
    if (params->gradient_mode == 2 || params->gradient_mode == 4) return DART_E_UNSUPPORTED;
    /* the promise of warm == 2 (zero lateral thrust) does not hold in the dynamics-consistent mode */
    if (params->gradient_mode == 3 && warm == 2) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.ld = ld;
    a.p0 = p; a.v0 = v; a.goal = goal; a.has_goal = has_goal;
    a.x_warm = warm ? x : nullptr;
    a.no_tilt_promise = (warm == 2) ? 1 : 0;
    a.x_out = x; a.cost = cost; a.nit = nit; a.nfev = nfev; a.status = status;
    a.p_next = p; a.v_next = v; a.plant_dt = plant_dt;
    return launch_solve(params, a, cuda_stream);
}

static bool grid_ok(const dart_grid *g)
{
    return g && g->occ && g->nx > 0 && g->ny > 0 && g->nz > 0 && g->resolution > 0.0 &&
           (g->cell_bytes == 0 || g->cell_bytes == 4 || g->cell_bytes == 8);
}

/* the step of dart_se3mpc_closed_loop_step_map (spheres == NULL) and
 * dart_se3mpc_closed_loop_step_spheres */
static int closed_loop_step_impl(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p, double *v,
                                 const double *goal, const uint8_t *has_goal, double *x, int32_t warm,
                                 double *cost, int32_t *nit, int32_t *nfev, int32_t *status, double plant_dt,
                                 const dart_grid *penalty_grid, const dart_spheres *spheres,
                                 const dart_grid *check_grid, double margin, double threshold, int32_t step,
                                 int32_t *first_collision, void *cuda_stream, const dart_track_ref *ref = nullptr,
                                 bool track = false)
{
    int rc = check_params(params, spheres != nullptr, track);
    if (rc) return rc;
    if (track && (rc = check_track(params, ref, spheres))) return rc;
    if (!track && spheres && (rc = check_spheres(spheres))) return rc;
    if (B < 0 || ld < B || !p || !v || (!goal && !track) || !x || !(plant_dt > 0.0)) return DART_E_BADARG;
    /* the reference window slides one sample per replan: one plant step must be one sample */
    if (track && plant_dt != params->dt) return DART_E_BADARG;
    const bool penalty = params->gradient_mode == 2 || params->gradient_mode == 4;
    if (penalty && !grid_ok(penalty_grid)) return DART_E_BADARG;
    if ((check_grid != nullptr) != (first_collision != nullptr)) return DART_E_BADARG;
    if (check_grid && !grid_ok(check_grid)) return DART_E_BADARG;
    /* the promise of warm == 2 (zero lateral thrust) does not hold in the dynamics-consistent modes */
    if (rollout_mode(params->gradient_mode) && warm == 2) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.ld = ld;
    a.p0 = p; a.v0 = v; a.goal = goal; a.has_goal = has_goal;
    a.x_warm = warm ? x : nullptr;
    a.no_tilt_promise = (warm == 2) ? 1 : 0;
    a.x_out = x; a.cost = cost; a.nit = nit; a.nfev = nfev; a.status = status;
    a.p_next = p; a.v_next = v; a.plant_dt = plant_dt;
    if (penalty) a.grid = *penalty_grid;
    if (check_grid) {
        a.check_grid = *check_grid;
        a.margin = margin;
        a.threshold = threshold;
        a.first_collision = first_collision;
        a.step = step;
    }
    set_spheres(a, spheres);
    set_track(a, ref);
    return launch_solve(params, a, cuda_stream);
}

int dart_se3mpc_closed_loop_step_map(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                     double *v, const double *goal, const uint8_t *has_goal, double *x,
                                     int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                     int32_t *status, double plant_dt, const dart_grid *penalty_grid,
                                     const dart_grid *check_grid, double margin, double threshold,
                                     int32_t step, int32_t *first_collision, void *cuda_stream)
{
    return closed_loop_step_impl(params, B, ld, p, v, goal, has_goal, x, warm, cost, nit, nfev, status, plant_dt,
                                 penalty_grid, nullptr, check_grid, margin, threshold, step, first_collision,
                                 cuda_stream);
}

int dart_se3mpc_closed_loop_step_spheres(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                         double *v, const double *goal, const uint8_t *has_goal, double *x,
                                         int32_t warm, double *cost, int32_t *nit, int32_t *nfev,
                                         int32_t *status, double plant_dt, const dart_spheres *spheres,
                                         const dart_grid *check_grid, double margin, double threshold,
                                         int32_t step, int32_t *first_collision, void *cuda_stream)
{
    if (!spheres) return DART_E_BADARG;
    return closed_loop_step_impl(params, B, ld, p, v, goal, has_goal, x, warm, cost, nit, nfev, status, plant_dt,
                                 nullptr, spheres, check_grid, margin, threshold, step, first_collision,
                                 cuda_stream);
}

int dart_se3mpc_solve_batch_track(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                  const double *p0, const double *v0, const uint8_t *has_goal,
                                  const double *x_warm, const uint8_t *warm_mask, double *x_out, double *cost,
                                  int32_t *nit, int32_t *nfev, int32_t *status, int32_t *task, double *acc,
                                  double *att, double *rates, double *thrust, const dart_track_ref *ref,
                                  const dart_spheres *spheres, const dart_grid *grid, double margin,
                                  double threshold, int32_t *first_hit, void *cuda_stream)
{
    return solve_batch_impl(params, B, ld, p0, v0, nullptr, has_goal, x_warm, warm_mask, x_out, cost, nit, nfev,
                            status, task, acc, att, rates, thrust, grid, margin, threshold, first_hit, spheres,
                            cuda_stream, ref, true);
}

int dart_se3mpc_closed_loop_step_track(const dart_se3mpc_params *params, int64_t B, int64_t ld, double *p,
                                       double *v, const uint8_t *has_goal, double *x, int32_t warm, double *cost,
                                       int32_t *nit, int32_t *nfev, int32_t *status, double plant_dt,
                                       const dart_track_ref *ref, const dart_spheres *spheres,
                                       const dart_grid *check_grid, double margin, double threshold,
                                       int32_t step, int32_t *first_collision, void *cuda_stream)
{
    return closed_loop_step_impl(params, B, ld, p, v, nullptr, has_goal, x, warm, cost, nit, nfev, status, plant_dt,
                                 nullptr, spheres, check_grid, margin, threshold, step, first_collision,
                                 cuda_stream, ref, true);
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

int dart_se3mpc_solve_batch_rows(const dart_se3mpc_params *params, int64_t B, int64_t ld,
                                 const double *p0, const double *v0, const double *goal,
                                 const uint8_t *has_goal, const double *x_warm,
                                 const uint8_t *warm_mask, double *rows, int64_t row_stride,
                                 int32_t row_kind, const dart_grid *grid, double margin,
                                 double threshold, int32_t check_map, void *cuda_stream)
{
    int rc = check_params(params);
    if (rc) return rc;
    if (B < 0 || ld < B || !p0 || !v0 || !goal || !rows) return DART_E_BADARG;
    if (row_kind < 0 || row_kind > 2) return DART_E_BADARG;
    if (row_kind == 1 && check_map) return DART_E_UNSUPPORTED; /* controls rows carry no map check */
    const int need = row_stride_doubles(params->horizon, row_kind);
    if (need == 0) return DART_E_UNSUPPORTED; /* the row does not fit its staging block */
    if (row_stride < need || (row_stride & 15) != 0 || row_stride > SM_DOUBLES ||
        ((uintptr_t)rows & 127) != 0)
        return DART_E_BADARG;
    const bool need_grid = check_map != 0 || params->gradient_mode == 2 || params->gradient_mode == 4;
    if (need_grid && (!grid || !grid->occ || grid->nx <= 0 || grid->ny <= 0 || grid->nz <= 0 ||
                      !(grid->resolution > 0.0)))
        return DART_E_BADARG;
    if (B == 0) return DART_OK;
    SolveArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.ld = ld;
    a.p0 = p0; a.v0 = v0; a.goal = goal; a.has_goal = has_goal;
    a.x_warm = x_warm; a.warm_mask = warm_mask;
    a.rows = rows; a.row_stride = row_stride; a.rows_kind = row_kind;
    if (need_grid) a.grid = a.check_grid = *grid;
    if (check_map) {
        a.margin = margin;
        a.threshold = threshold;
        a.check_map = 1; /* the result goes into the row */
    }
    return launch_solve(params, a, cuda_stream);
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

/* workspace layout for row pitch Bp (elements): fp64 rows [p0 3 | v0 3 | goal 3 | x_warm 9N |
 * x 9N | cost 1 | acc 3N | att 3N | rates 3N | thrust N], int32 rows [nit nfev status task],
 * u8 row [has_goal].  Inputs are one contiguous range, outputs another. */
struct WsLayout {
    size_t Bp, in_rows, out_off_rows, out_rows, int_off, hg_off, bytes;
    WsLayout(int N, size_t Bp_) : Bp(Bp_)
    {
        in_rows = 9 + 9 * (size_t)N;
        out_off_rows = in_rows;
        out_rows = 9 * (size_t)N + 1 + 9 * (size_t)N + (size_t)N;
        int_off = (in_rows + out_rows) * Bp * 8;
        hg_off = int_off + 4 * Bp * 4;
        bytes = hg_off + ((Bp + 7) / 8) * 8;
    }
};

void rows_in(void *dst, size_t pitch, const void *src, size_t B, size_t rows, size_t esz)
{
    for (size_t r = 0; r < rows; ++r)
        memcpy((char *)dst + r * pitch * esz, (const char *)src + r * B * esz, B * esz);
}
void rows_out(void *dst, const void *src, size_t pitch, size_t B, size_t rows, size_t esz)
{
    if (!dst) return;
    for (size_t r = 0; r < rows; ++r)
        memcpy((char *)dst + r * B * esz, (const char *)src + r * pitch * esz, B * esz);
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

/* the host entry of dart_se3mpc_solve_batch_host (spheres == NULL) and
 * dart_se3mpc_solve_batch_host_spheres (the list in host memory: staged behind the workspace) */
static int solve_batch_host_impl(const dart_se3mpc_params *params, int64_t B, const double *p0, const double *v0,
                                 const double *goal, const uint8_t *has_goal, const double *x_warm,
                                 double *x_out, double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                                 double *acc, double *att, double *rates, double *thrust,
                                 const dart_spheres *spheres)
{
    int rc = check_params(params, spheres != nullptr);
    if (rc) return rc;
    if (spheres && (rc = check_spheres(spheres))) return rc;
    if (B < 0 || !p0 || !v0 || !goal) return DART_E_BADARG;
    if (B == 0) return DART_OK;
    const size_t N = (size_t)params->horizon;
    /* small batches (the drop-in planner's single solve): no copies at all -- the kernel reads its
     * inputs from and writes its results to a mapped pinned block over PCIe (zero-copy: one
     * launch and one synchronise; 62 us instead of 85 us at 512 problems); large batches copy
     * rows straight from / to the caller's buffers */
    const bool staged = B <= 512;
    const size_t Bp = staged ? (size_t)((B + 3) / 4 * 4) : (size_t)((B + 31) / 32 * 32);
    const WsLayout L((int)N, Bp);
    /* the sphere list, if any, follows the workspace: [n][4] doubles at a 16-byte offset */
    const size_t sph_off = (L.bytes + 15) / 16 * 16;
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
    double *d = (double *)base;
    double *d_p0 = d, *d_v0 = d_p0 + 3 * Bp, *d_goal = d_v0 + 3 * Bp, *d_xw = d_goal + 3 * Bp;
    double *d_x = d_xw + 9 * N * Bp, *d_cost = d_x + 9 * N * Bp;
    double *d_acc = d_cost + Bp, *d_att = d_acc + 3 * N * Bp, *d_rates = d_att + 3 * N * Bp;
    double *d_thr = d_rates + 3 * N * Bp;
    int32_t *d_nit = (int32_t *)(base + L.int_off), *d_nfev = d_nit + Bp, *d_status = d_nfev + Bp,
            *d_task = d_status + Bp;
    uint8_t *d_hg = (uint8_t *)(base + L.hg_off);
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
    const dart_spheres *dsp = spheres ? &dsph : nullptr;
    if (!staged && B >= 65536) {
        /* Large batch: chunks of 32768 problems alternate between two streams, each doing its own
         * pitched H2D rows -> solve -> pitched D2H rows, so the read-back of chunk i (the
         * dominant cost: 1.3 KB per solve over PCIe) overlaps the solve of chunk i+1 and the
         * upload of chunk i+2.  Fully asynchronous when the caller's buffers are pinned. */
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
        const int64_t chunk = 32768;
        int ci = 0;
        /* on a failure mid-loop the copies already queued still write into the caller's buffers:
         * wait for them before handing the buffers back */
        auto drain = [&]() {
            cudaStreamSynchronize(g_ws.stream);
            cudaStreamSynchronize(g_ws.stream2);
        };
        struct HintScope { /* every chunk runs the build chosen for the whole batch */
            explicit HintScope(long long b) { g_batch_hint = b; }
            ~HintScope() { g_batch_hint = 0; }
        } hint_scope(B);
        for (int64_t c0 = 0; c0 < B; c0 += chunk, ++ci) {
            const int64_t cb = (B - c0 < chunk) ? (B - c0) : chunk;
            cudaStream_t cs = (ci & 1) ? g_ws.stream2 : g_ws.stream;
#define ROWS_H2D(dst, src, rows, esz)                                                                        \
    do {                                                                                                     \
        e = cudaMemcpy2DAsync((char *)(dst) + c0 * (esz), Bp * (esz), (const char *)(src) + c0 * (esz),        \
                              (size_t)B * (esz), (size_t)cb * (esz), rows, cudaMemcpyHostToDevice, cs);       \
        if (e != cudaSuccess) return drain(), set_err(e, "cudaMemcpy2DAsync H2D");                           \
    } while (0)
#define ROWS_D2H(dst, src, rows, esz)                                                                        \
    do {                                                                                                     \
        if (dst) {                                                                                           \
            e = cudaMemcpy2DAsync((char *)(dst) + c0 * (esz), (size_t)B * (esz), (const char *)(src) + c0 * (esz), \
                                  Bp * (esz), (size_t)cb * (esz), rows, cudaMemcpyDeviceToHost, cs);          \
            if (e != cudaSuccess) return drain(), set_err(e, "cudaMemcpy2DAsync D2H");                       \
        }                                                                                                    \
    } while (0)
            ROWS_H2D(d_p0, p0, 3, 8);
            ROWS_H2D(d_v0, v0, 3, 8);
            ROWS_H2D(d_goal, goal, 3, 8);
            if (has_goal) ROWS_H2D(d_hg, has_goal, 1, 1);
            if (x_warm) ROWS_H2D(d_xw, x_warm, 9 * N, 8);
            rc = solve_batch_impl(params, cb, (int64_t)Bp, d_p0 + c0, d_v0 + c0, d_goal + c0,
                                  has_goal ? d_hg + c0 : nullptr, x_warm ? d_xw + c0 : nullptr, nullptr,
                                  x_out ? d_x + c0 : nullptr, cost ? d_cost + c0 : nullptr,
                                  nit ? d_nit + c0 : nullptr, nfev ? d_nfev + c0 : nullptr,
                                  status ? d_status + c0 : nullptr, nullptr, acc ? d_acc + c0 : nullptr,
                                  att ? d_att + c0 : nullptr, rates ? d_rates + c0 : nullptr,
                                  thrust ? d_thr + c0 : nullptr, nullptr, 0.0, 0.0, nullptr, dsp, (void *)cs);
            if (rc) return drain(), rc;
            ROWS_D2H(x_out, d_x, 9 * N, 8);
            ROWS_D2H(cost, d_cost, 1, 8);
            ROWS_D2H(nit, d_nit, 1, 4);
            ROWS_D2H(nfev, d_nfev, 1, 4);
            ROWS_D2H(status, d_status, 1, 4);
            ROWS_D2H(acc, d_acc, 3 * N, 8);
            ROWS_D2H(att, d_att, 3 * N, 8);
            ROWS_D2H(rates, d_rates, 3 * N, 8);
            ROWS_D2H(thrust, d_thr, N, 8);
#undef ROWS_H2D
#undef ROWS_D2H
        }
        e = cudaStreamSynchronize(g_ws.stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(g_ws.stream2);
        if (e != cudaSuccess) return set_err(e, "cudaStreamSynchronize");
        return DART_OK;
    }
    if (staged) {
        char *h = (char *)g_ws.pin;
        rows_in(h, Bp, p0, (size_t)B, 3, 8);
        rows_in(h + 3 * Bp * 8, Bp, v0, (size_t)B, 3, 8);
        rows_in(h + 6 * Bp * 8, Bp, goal, (size_t)B, 3, 8);
        if (x_warm) rows_in(h + 9 * Bp * 8, Bp, x_warm, (size_t)B, 9 * N, 8);
        if (has_goal) memcpy(h + L.hg_off, has_goal, (size_t)B);
    } else {
#define H2D(dst, src, rows, esz)                                                              \
    do {                                                                                      \
        e = cudaMemcpy2DAsync(dst, Bp * (esz), src, (size_t)B * (esz), (size_t)B * (esz), rows, \
                              cudaMemcpyHostToDevice, s);                                     \
        if (e != cudaSuccess) return set_err(e, "cudaMemcpy2DAsync H2D");                     \
    } while (0)
        H2D(d_p0, p0, 3, 8);
        H2D(d_v0, v0, 3, 8);
        H2D(d_goal, goal, 3, 8);
        if (has_goal) H2D(d_hg, has_goal, 1, 1);
        if (x_warm) H2D(d_xw, x_warm, 9 * N, 8);
#undef H2D
    }
    const bool all = false; /* only the rows the caller asked for are computed and written */
    rc = solve_batch_impl(params, B, (int64_t)Bp, d_p0, d_v0, d_goal, has_goal ? d_hg : nullptr,
                          x_warm ? d_xw : nullptr, nullptr, (all || x_out) ? d_x : nullptr,
                          (all || cost) ? d_cost : nullptr, (all || nit) ? d_nit : nullptr,
                          (all || nfev) ? d_nfev : nullptr, (all || status) ? d_status : nullptr,
                          nullptr, (all || acc) ? d_acc : nullptr, (all || att) ? d_att : nullptr,
                          (all || rates) ? d_rates : nullptr, (all || thrust) ? d_thr : nullptr,
                          nullptr, 0.0, 0.0, nullptr, dsp, (void *)s);
    if (rc) return rc;
    if (staged) {
        char *h = (char *)g_ws.pin;
        e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return set_err(e, "cudaStreamSynchronize");
        const double *hd = (const double *)h;
        const double *h_x = hd + L.in_rows * Bp, *h_cost = h_x + 9 * N * Bp, *h_acc = h_cost + Bp,
                     *h_att = h_acc + 3 * N * Bp, *h_rates = h_att + 3 * N * Bp, *h_thr = h_rates + 3 * N * Bp;
        const int32_t *h_nit = (const int32_t *)(h + L.int_off);
        rows_out(x_out, h_x, Bp, (size_t)B, 9 * N, 8);
        rows_out(cost, h_cost, Bp, (size_t)B, 1, 8);
        rows_out(acc, h_acc, Bp, (size_t)B, 3 * N, 8);
        rows_out(att, h_att, Bp, (size_t)B, 3 * N, 8);
        rows_out(rates, h_rates, Bp, (size_t)B, 3 * N, 8);
        rows_out(thrust, h_thr, Bp, (size_t)B, N, 8);
        rows_out(nit, h_nit, Bp, (size_t)B, 1, 4);
        rows_out(nfev, h_nit + Bp, Bp, (size_t)B, 1, 4);
        rows_out(status, h_nit + 2 * Bp, Bp, (size_t)B, 1, 4);
        return DART_OK;
    }
#define D2H(dst, src, rows, esz)                                                              \
    do {                                                                                      \
        if (dst) {                                                                            \
            e = cudaMemcpy2DAsync(dst, (size_t)B * (esz), src, Bp * (esz), (size_t)B * (esz), rows, \
                                  cudaMemcpyDeviceToHost, s);                                 \
            if (e != cudaSuccess) return set_err(e, "cudaMemcpy2DAsync D2H");                 \
        }                                                                                     \
    } while (0)
    D2H(x_out, d_x, 9 * N, 8);
    D2H(cost, d_cost, 1, 8);
    D2H(nit, d_nit, 1, 4);
    D2H(nfev, d_nfev, 1, 4);
    D2H(status, d_status, 1, 4);
    D2H(acc, d_acc, 3 * N, 8);
    D2H(att, d_att, 3 * N, 8);
    D2H(rates, d_rates, 3 * N, 8);
    D2H(thrust, d_thr, N, 8);
#undef D2H
    e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return set_err(e, "cudaStreamSynchronize");
    return DART_OK;
}

int dart_se3mpc_solve_batch_host(const dart_se3mpc_params *params, int64_t B,
                                 const double *p0, const double *v0, const double *goal,
                                 const uint8_t *has_goal, const double *x_warm, double *x_out,
                                 double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                                 double *acc, double *att, double *rates, double *thrust)
{
    return solve_batch_host_impl(params, B, p0, v0, goal, has_goal, x_warm, x_out, cost, nit, nfev, status, acc,
                                 att, rates, thrust, nullptr);
}

int dart_se3mpc_solve_batch_host_spheres(const dart_se3mpc_params *params, int64_t B,
                                         const double *p0, const double *v0, const double *goal,
                                         const uint8_t *has_goal, const double *x_warm, double *x_out,
                                         double *cost, int32_t *nit, int32_t *nfev, int32_t *status,
                                         double *acc, double *att, double *rates, double *thrust,
                                         const dart_spheres *spheres)
{
    if (!spheres) return DART_E_BADARG;
    return solve_batch_host_impl(params, B, p0, v0, goal, has_goal, x_warm, x_out, cost, nit, nfev, status, acc,
                                 att, rates, thrust, spheres);
}

} /* extern "C" */
