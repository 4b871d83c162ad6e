// C ABI of libarmour_b200.so (see include/armour_b200.h).  One translation unit: the kernels are
// included below so they share the __constant__ block.  No CPU fallback anywhere: every compute entry
// point launches CUDA kernels on the context's stream and reports CUDA errors as ARMOUR_ERR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/armour_b200.h"
#include "bezier.cuh"
#include "device_constants.cuh"
// The reach-set kernel is compiled twice (see k1_pz.cuh):
//   k1lat: one unit per CTA built by 3 groups of 128 threads (task list, MG mode) -> lowest latency for one planning problem
//   k1thr: 2 CTAs per SM of 8 units each in lock step, 64 threads per unit -> highest throughput for batches.  Instruction
//          fetch bounds this kernel: the units of a CTA run the same operation at the same time (without the lock step the
//          instruction cache thrashes: 2.3x slower), and two lock-step domains per SM overlap each other's barriers.  A unit
//          keeps only its control block in shared memory; arena, scratch and joint reachable set live in its global scratch,
//          behind the L1 cache that the unclaimed shared memory becomes (profiles/r3_k1thr_experiments.md: 445 -> 360 us
//          per problem; round-1 sweep with one CTA per SM: 8 groups 535 us, 10: 519, 12: 503, 14: 497)
#ifdef K1_PROFILE
constexpr int K1_PROF_SITES = 512;
__device__ long long g_k1prof[128 * K1_PROF_SITES * 2];
__device__ int g_k1spill[8];  // arena blocks in global memory, all arena blocks, scratch pools in global memory
#endif
// Latency configuration: MG mode, K1LAT_GROUPS groups of K1LAT_NT threads build ONE unit together (one CTA per SM)
#ifndef K1LAT_NT
#define K1LAT_NT 128
#endif
#ifndef K1LAT_CTAS
#define K1LAT_CTAS 1
#endif
#ifndef K1LAT_GROUPS
#define K1LAT_GROUPS 3
#endif
#ifndef K1LAT_MG
#define K1LAT_MG 1
#endif
#ifndef K1LAT_TAB_16THS
#define K1LAT_TAB_16THS 11  // share (in sixteenths) of a group's dynamic shared memory given to the scratch pool
#endif
#define K1_TAB_16THS K1LAT_TAB_16THS
#ifndef K1LAT_DYN_CAP
#define K1LAT_DYN_CAP -1  // shared memory per group beyond the fixed region: no cap
#endif
#define K1_DYN_CAP K1LAT_DYN_CAP
#define K1_NS k1lat
#define K1_NT K1LAT_NT
#define K1_CTAS K1LAT_CTAS
#define K1_GROUPS K1LAT_GROUPS
#define K1_MG K1LAT_MG
#include "k1_reachsets.cuh"
#undef K1_NS
#undef K1_NT
#undef K1_CTAS
#undef K1_GROUPS
#undef K1_MG
#undef K1_TAB_16THS
#define K1_MG 0
#ifndef K1THR_NT
#define K1THR_NT 64
#endif
#ifndef K1THR_GROUPS
#define K1THR_GROUPS 8
#endif
#ifndef K1THR_CTAS
#define K1THR_CTAS 2
#endif
#ifndef K1THR_TAB_EIGHTHS
#define K1THR_TAB_EIGHTHS 4  // share (in eighths) of a group's dynamic shared memory given to the scratch pool
#endif
#ifndef K1THR_DYN_CAP
#define K1THR_DYN_CAP 0  // no shared-memory arena / scratch per group: the global scratch behind a large L1 is faster (DESIGN.md section 6)
#endif
#ifndef K1THR_JRS_GLOBAL
#define K1THR_JRS_GLOBAL 1  // the joint-reachable-set region of a group sits in its global scratch too (only the control block in shared memory)
#endif
#undef K1_JRS_GLOBAL
#define K1_JRS_GLOBAL K1THR_JRS_GLOBAL
#undef K1_DYN_CAP
#define K1_DYN_CAP K1THR_DYN_CAP
#undef K1_TAB_EIGHTHS
#define K1_TAB_EIGHTHS K1THR_TAB_EIGHTHS
#define K1_TAB_16THS (2 * K1THR_TAB_EIGHTHS)
#define K1_NS k1thr
#define K1_NT K1THR_NT
#define K1_CTAS K1THR_CTAS
#define K1_GROUPS K1THR_GROUPS
#include "k1_reachsets.cuh"
#undef K1_NS
#undef K1_NT
#undef K1_CTAS
#undef K1_GROUPS
#include "k3_constraints.cuh"
#include "k4_solver.cuh"
#include "armtd.cuh"
#include "rollout.cuh"
#include "layout.h"
#include "device_buffer.h"

using namespace armour;

// Every device allocation of a context is one of its DeviceBuffer members (or K1Scratch's); the pointers of B are views of them.
struct armour_ctx {
    armour_config cfg;
    RobotConstants rc;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    Batch B;                 // device pointers + dimensions of the current batch
    int built_nprob = 0;     // problems with valid reach sets
    // reach-set tables of max_problems problems, allocated at creation (B.link_n ... B.status)
    DeviceBuffer<int> link_n, u_n, status;
    DeviceBuffer<double> link_c, link_g, u_c, u_r, u_g, torque_radius, link_gens, link_r, link_sliced;
    DeviceBuffer<uint16_t> link_key, u_key;
    // sized for the batch by ensure_obstacle_buffers (B.obstacles, B.img, B.hp_cnt, B.hp_slow)
    DeviceBuffer<double> d_obs;
    DeviceBuffer<unsigned char> img, hp_cnt;
    DeviceBuffer<int> hp_slow;
    DeviceBuffer<int> d_unit_flag;  // [max_problems * T] completion stamps of the reach-set units (latency path)
    DeviceBuffer<double> d_in;      // [3][max_problems][NF] q0, qd0, qdd0
    DeviceBuffer<double> d_k;       // staging for the host-pointer evaluation calls
    DeviceBuffer<double> d_g, d_jac;
    DeviceBuffer<double> d_jnz;     // packed non-zeros of the Jacobian (structured evaluation)
    DeviceBuffer<int> d_verdict;    // [2][max_problems]
    // batched device solver (allocated on first use)
    DeviceBuffer<double> d_solver;  // state arrays + second g buffer + linearised rows
    DeviceBuffer<int> d_solver_i;   // have_best, status, iters, evals, running counter
    k1lat::K1Scratch k1_lat;  // scratch of the latency configuration of k_reachsets
    k1thr::K1Scratch k1_thr;  // scratch of the throughput configuration (allocated on first use)
    bool k1_thr_ready = false;
    long long launches = 0;
    std::string last_error;
    std::vector<double> h_torque_radius;  // host mirror of problem 0..built_nprob-1 (lazy)
    bool h_torque_valid = false;
    std::vector<double> h_q0, h_qd0, h_qdd0;
    // ARMTD comparison planner (armour_armtd_*): imported joint reachable set, KPA-layout outputs, trajectory parameters
    bool armtd = false;
    DeviceBuffer<double> d_jrs;       // [max_problems][ARMTD_T_PADDED][NF][6] the offline table rotated by q0 (B.jrs_ext)
    DeviceBuffer<double> d_armtd_in;  // one allocation for the four arrays below
    double* d_krange = nullptr;    // [max_problems][NF] k_range of each problem
    double* d_zero = nullptr;      // [max_problems][NF] zeros: qdd0 of the build (unused by the forward kinematics)
    double* d_cs = nullptr;        // [max_problems][NF][2] cos q0, sin q0 staged by the host-pointer build
    double* d_jrs_raw = nullptr;   // [max_problems][6][NF][ARMTD_T] offline tables staged by the host-pointer build
    DeviceBuffer<double> d_ga;     // [nprob][m_armtd] KPA-layout g of the host-pointer calls and of the solver
    DeviceBuffer<double> d_ja;     // [nprob][m_armtd][NF]
    std::vector<double> h_krange;  // host mirror of d_krange for the cost (empty: fetched after a device build)
    // closed-loop episodes (armour_batch_rollout*), allocated on first use
    DeviceBuffer<double> d_roll;  // per-world state, current plans and the dense batch of a rollout
    DeviceBuffer<int> d_roll_i;   // outcomes, counters, world lists, verdicts
    DeviceBuffer<char> d_stage;   // inputs and outputs of the host-pointer calls that stage (see stage())
};

namespace {

// FP64 FMA throughput probe: 8 independent accumulator chains per thread
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double a) {
    double x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = double(threadIdx.x + i);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 8; i++) x[i] = __fma_rn(x[i], a, 0.5);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) s += x[i];
    if (s == 12345.678) out[0] = s;  // never true; keeps the chains alive
}

int fail(armour_ctx* c, int code, const std::string& msg) {
    if (c) c->last_error = msg;
    return code;
}
#define CU(expr)                                                                                     \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return fail(ctx, ARMOUR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
    } while (0)

// d_g / d_jac for `rows` constraint rows (of all problems together)
int ensure_eval_buffers(armour_ctx* ctx, size_t rows, bool need_g, bool need_jac) {
    if (need_g) CU(ctx->d_g.reserve(rows));
    if (need_jac) CU(ctx->d_jac.reserve(rows * NF));
    return ARMOUR_OK;
}

// The obstacle, image and candidate-count buffers of a batch of nprob problems with nobs obstacles each.  The current batch
// (B.O, B.nprob) is the caller's to set.
int ensure_obstacle_buffers(armour_ctx* ctx, int nprob, int nobs) {
    Batch& B = ctx->B;
    Batch next = B;
    next.O = nobs;
    const size_t need_img = size_t(nprob) * (B.T / TB) * next.img_chunk();
    const size_t need_cnt = size_t(nprob) * B.T * B.NJ * nobs;
    const bool regrow = ctx->img.capacity() < need_img || ctx->hp_cnt.capacity() < need_cnt || ctx->hp_slow.capacity() < size_t(nprob);
    // growing drops the built batch: its candidate lists and images go with the old buffers.  (The obstacle buffer grows only
    // when hp_cnt does, so a batch whose obstacles were freed is never left built either.)
    if (regrow) ctx->built_nprob = 0;
    CU(ctx->d_obs.reserve(size_t(nprob) * nobs * 12));
    B.obstacles = ctx->d_obs.get();
    if (regrow) {
        ctx->img = {};
        ctx->hp_cnt = {};
        ctx->hp_slow = {};
        CU(ctx->img.reserve(need_img));
        CU(ctx->hp_cnt.reserve(std::max<size_t>(need_cnt, 1)));  // (one byte without obstacles: B.hp_cnt is never null)
        CU(ctx->hp_slow.reserve(nprob));
        CU(cudaMemsetAsync(ctx->hp_slow.get(), 0, nprob * sizeof(int), ctx->stream));
        B.img = ctx->img.get();
        B.hp_cnt = ctx->hp_cnt.get();
        B.hp_slow = ctx->hp_slow.get();
    }
    return ARMOUR_OK;
}

// Pick the kernel configuration by batch size: up to two waves of the latency configuration's CTAs are
// faster there; beyond that the lock-step throughput configuration wins (DESIGN.md, K1).
int launch_build(armour_ctx* ctx, const Batch& B, int* nl, bool* latency) {
    const long long nunits = (long long)B.nprob * B.T;
    const bool thr = ctx->cfg.max_problems > 1 && nunits > 2LL * ctx->k1_lat.grid;
    *latency = !thr;
    if (thr) {
        if (!ctx->k1_thr_ready) {
            CU(k1thr::k1_scratch_create(&ctx->k1_thr, ctx->cfg, ctx->rc, ctx->stream));
            ctx->k1_thr_ready = true;
        }
        CU(k1thr::launch_reachsets(B, ctx->k1_thr, ctx->stream, nl));
    } else {
        CU(k1lat::launch_reachsets(B, ctx->k1_lat, ctx->stream, nl, ctx->d_unit_flag.get()));
    }
    return ARMOUR_OK;
}

// The robot / planner constants live in ONE __constant__ block per device, shared by every context of the process.
// Before a context launches anything it makes sure the block holds ITS constants: contexts with identical
// configurations share the block freely; switching between contexts that differ (gripper model, threshold, k_range,
// uncertainties ...) waits for the device to drain and uploads again, so no kernel ever runs on another context's
// constants.  (Correct, not fast: interleave differing contexts on one device sparingly.)
std::mutex g_const_mutex;
struct ConstOwner {
    bool valid = false;
    RobotConstants rc;
};
ConstOwner g_const_owner[64];

int ensure_constants(armour_ctx* ctx) {
    const int dev = ctx->cfg.device;
    if (dev < 0 || dev >= 64) return fail(ctx, ARMOUR_ERR_ARG, "device ordinal");
    std::lock_guard<std::mutex> lock(g_const_mutex);
    ConstOwner& o = g_const_owner[dev];
    if (o.valid && std::memcmp(&o.rc, &ctx->rc, sizeof(RobotConstants)) == 0) return ARMOUR_OK;
    CU(cudaDeviceSynchronize());  // kernels of the previous owner may still read the block
    CU(upload_constants(ctx->rc, ctx->stream));
    o.rc = ctx->rc;
    o.valid = true;
    return ARMOUR_OK;
}

// First step of an entry point that launches: this context's device, and its constants on that device.
int enter(armour_ctx* ctx) {
    CU(cudaSetDevice(ctx->cfg.device));
    return ensure_constants(ctx);
}

// The host-pointer calls that stage their inputs and outputs cut the context's one staging buffer into pieces of the given
// sizes in bytes, 256-byte aligned (nullptr for a size of 0).  A call that stages may call only *_device entry points: any
// other host-pointer call could stage over its pieces.
template <size_t N>
int stage(armour_ctx* ctx, const size_t (&bytes)[N], void* (&piece)[N]) {
    size_t total = 0;
    for (size_t b : bytes) total += (b + 255) / 256 * 256;
    CU(ctx->d_stage.reserve(total));
    char* p = ctx->d_stage.get();
    for (size_t i = 0; i < N; i++) {
        piece[i] = bytes[i] ? p : nullptr;
        p += (bytes[i] + 255) / 256 * 256;
    }
    return ARMOUR_OK;
}

int check_batch(armour_ctx* ctx, int nprob, int nobs) {
    if (!ctx) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->cfg.max_problems)
        return fail(ctx, ARMOUR_ERR_STATE, "nprob outside [1, max_problems]");
    if (nobs < 0) return fail(ctx, ARMOUR_ERR_ARG, "negative obstacle count");
    if (nobs > ctx->cfg.max_obstacles)
        return fail(ctx, ARMOUR_ERR_OBSTACLES, "number of obstacles larger than max_obstacles");
    return ARMOUR_OK;
}

int fetch_torque_radius(armour_ctx* ctx) {
    if (ctx->h_torque_valid) return ARMOUR_OK;
    const size_t n = size_t(ctx->built_nprob) * NF * ctx->B.T;
    ctx->h_torque_radius.resize(n);
    CU(cudaMemcpyAsync(ctx->h_torque_radius.data(), ctx->B.torque_radius, n * sizeof(double), cudaMemcpyDeviceToHost,
                       ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    ctx->h_torque_valid = true;
    return ARMOUR_OK;
}

}  // namespace

extern "C" {

int armour_abi_version(void) { return ARMOUR_ABI_VERSION; }

const char* armour_status_string(int s) {
    switch (s) {
        case ARMOUR_OK: return "ok";
        case ARMOUR_ERR_ARG: return "invalid argument";
        case ARMOUR_ERR_CUDA: return "CUDA error";
        case ARMOUR_ERR_OBSTACLES: return "too many obstacles";
        case ARMOUR_ERR_CAPACITY: return "monomial table capacity exceeded";
        case ARMOUR_ERR_STATE: return "invalid call order or batch size";
        case ARMOUR_ERR_NOMEM: return "out of memory";
        default: return "unknown status";
    }
}

int armour_config_default(armour_config* cfg) {
    if (!cfg) return ARMOUR_ERR_ARG;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->struct_size = int(sizeof(armour_config));
    cfg->device = 0;
    cfg->robot_model = 0;
    cfg->num_time_steps = 128;
    cfg->max_obstacles = 40;
    cfg->max_problems = 1;
    cfg->cap_link_monomials = 32;
    cfg->cap_torque_monomials = 64;
    cfg->cap_work_monomials = 768;
    cfg->simplify_threshold = 5e-4;
    for (int i = 0; i < NF; i++) cfg->k_range[i] = M_PI / 48;
    cfg->mass_uncertainty = -1;
    cfg->inertia_uncertainty = -1;
    return ARMOUR_OK;
}

int armour_ctx_create(const armour_config* cfg, armour_ctx** out) {
    if (!cfg || !out) return ARMOUR_ERR_ARG;
    *out = nullptr;
    if (cfg->struct_size != int(sizeof(armour_config))) return ARMOUR_ERR_ARG;
    if (cfg->num_time_steps < TB || cfg->num_time_steps > 128 || cfg->num_time_steps % TB != 0) return ARMOUR_ERR_ARG;
    if (cfg->max_problems < 1 || cfg->max_obstacles < 0) return ARMOUR_ERR_ARG;
    if (cfg->robot_model < 0 || cfg->robot_model > 1) return ARMOUR_ERR_ARG;
    if (cfg->cap_link_monomials < 1 || cfg->cap_torque_monomials < 1 || cfg->cap_work_monomials < 64)
        return ARMOUR_ERR_ARG;
    // the stored tables are fetched with 16-byte bulk copies (keys are 2 bytes): capacities in multiples of 8
    if (cfg->cap_link_monomials % 8 != 0 || cfg->cap_torque_monomials % 8 != 0) return ARMOUR_ERR_ARG;
    if (cfg->max_problems > 65535) return ARMOUR_ERR_ARG;  // the problem index is gridDim.y of the constraint kernels
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg->device >= ndev) return ARMOUR_ERR_CUDA;
    armour_ctx* ctx = new (std::nothrow) armour_ctx();
    if (!ctx) return ARMOUR_ERR_NOMEM;
    ctx->cfg = *cfg;
    ctx->rc = make_robot_constants(cfg->robot_model);
    ctx->rc.num_time_steps = cfg->num_time_steps;
    ctx->rc.simplify_threshold = cfg->simplify_threshold;
    for (int i = 0; i < NF; i++) ctx->rc.k_range[i] = cfg->k_range[i];
    if (cfg->mass_uncertainty >= 0) ctx->rc.mass_uncertainty = cfg->mass_uncertainty;
    if (cfg->inertia_uncertainty >= 0) ctx->rc.inertia_uncertainty = cfg->inertia_uncertainty;

    auto bail = [&](const char* what, cudaError_t e) {
        std::fprintf(stderr, "armour_ctx_create: %s: %s\n", what, cudaGetErrorString(e));
        armour_ctx_destroy(ctx);
        return ARMOUR_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) return bail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess)
        return bail("cudaStreamCreate", e);
    ctx->stream = ctx->own_stream;
    if (ensure_constants(ctx) != ARMOUR_OK) return bail("upload_constants", cudaGetLastError());

    Batch& B = ctx->B;
    std::memset(&B, 0, sizeof(B));
    B.T = cfg->num_time_steps;
    B.NJ = ctx->rc.num_joints;
    B.capL = cfg->cap_link_monomials;
    B.capU = cfg->cap_torque_monomials;
    const size_t P = size_t(cfg->max_problems), T = size_t(B.T), NJ = size_t(B.NJ);
#define ALLOC(buf, n) \
    if ((e = ctx->buf.reserve(n)) != cudaSuccess) return bail(#buf, e)
#define TABLE(field, n) \
    ALLOC(field, n);    \
    B.field = ctx->field.get()
    ALLOC(d_in, 3 * P * NF);
    TABLE(link_n, P * T * NJ);
    TABLE(link_c, P * T * NJ * 3);
    TABLE(link_key, P * T * NJ * B.capL);
    TABLE(link_g, P * T * NJ * B.capL * 3);
    TABLE(u_n, P * T * NF);
    TABLE(u_c, P * T * NF);
    TABLE(u_r, P * T * NF);
    TABLE(u_key, P * T * NF * B.capU);
    TABLE(u_g, P * T * NF * B.capU);
    TABLE(torque_radius, P * NF * T);
    TABLE(link_gens, P * T * NJ * 18);
    TABLE(link_r, P * T * NJ * 3);
    TABLE(link_sliced, P * T * NJ * 3);
    TABLE(status, P);
    ALLOC(d_unit_flag, P * T);
    ALLOC(d_k, P * NF);
    ALLOC(d_verdict, 2 * P);
#undef TABLE
#undef ALLOC
    B.q0 = ctx->d_in.get();
    B.qd0 = ctx->d_in.get() + P * NF;
    B.qdd0 = ctx->d_in.get() + 2 * P * NF;
    if ((e = cudaMemsetAsync(B.status, 0, P * sizeof(int), ctx->stream)) != cudaSuccess) return bail("memset", e);
    if ((e = cudaMemsetAsync(ctx->d_unit_flag.get(), 0, P * T * sizeof(int), ctx->stream)) != cudaSuccess) return bail("memset", e);
    // no table may ever be read with an uninitialised count (a failed build leaves its tables untouched)
    if ((e = cudaMemsetAsync(B.link_n, 0, P * T * NJ * sizeof(int), ctx->stream)) != cudaSuccess) return bail("memset", e);
    if ((e = cudaMemsetAsync(B.u_n, 0, P * T * NF * sizeof(int), ctx->stream)) != cudaSuccess) return bail("memset", e);
    if ((e = k1lat::k1_scratch_create(&ctx->k1_lat, ctx->cfg, ctx->rc, ctx->stream)) != cudaSuccess) return bail("k1 scratch", e);
    if ((long long)cfg->max_problems * B.T > 2LL * ctx->k1_lat.grid) {  // this context can see batches: set up the throughput kernel too
        if ((e = k1thr::k1_scratch_create(&ctx->k1_thr, ctx->cfg, ctx->rc, ctx->stream)) != cudaSuccess) return bail("k1 throughput scratch", e);
        ctx->k1_thr_ready = true;
        cudaFuncAttributes fa2;
        if ((e = cudaFuncGetAttributes(&fa2, k1thr::k_reachsets)) != cudaSuccess) return bail("load k_reachsets (throughput)", e);
    }
    {   // load the kernels now (CUDA loads modules lazily at first use), so that the first build is not charged for it
        cudaFuncAttributes fa;
        if ((e = cudaFuncGetAttributes(&fa, k1lat::k_reachsets)) != cudaSuccess) return bail("load k_reachsets", e);
        if ((e = cudaFuncGetAttributes(&fa, k_hyperplanes)) != cudaSuccess) return bail("load k_hyperplanes", e);
        if ((e = cudaFuncGetAttributes(&fa, k_constraints)) != cudaSuccess) return bail("load k_constraints", e);
        if ((e = cudaFuncGetAttributes(&fa, k_constraints_slow)) != cudaSuccess) return bail("load k_constraints_slow", e);
        if ((e = cudaFuncGetAttributes(&fa, k_verdict)) != cudaSuccess) return bail("load k_verdict", e);
    }
    if ((e = cudaStreamSynchronize(ctx->stream)) != cudaSuccess) return bail("sync", e);
    *out = ctx;
    return ARMOUR_OK;
}

int armour_ctx_destroy(armour_ctx* ctx) {
    if (!ctx) return ARMOUR_OK;
    cudaSetDevice(ctx->cfg.device);
    k1lat::k1_scratch_destroy(&ctx->k1_lat);
    k1thr::k1_scratch_destroy(&ctx->k1_thr);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;  // frees the buffers
    return ARMOUR_OK;
}

int armour_ctx_set_stream(armour_ctx* ctx, void* s) {
    if (!ctx) return ARMOUR_ERR_ARG;
    ctx->stream = s ? static_cast<cudaStream_t>(s) : ctx->own_stream;
    return ARMOUR_OK;
}
int armour_ctx_synchronize(armour_ctx* ctx) {
    if (!ctx) return ARMOUR_ERR_ARG;
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}
const char* armour_last_error(const armour_ctx* ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
long long armour_kernel_launches(const armour_ctx* ctx) { return ctx ? ctx->launches : 0; }
int armour_num_joints(const armour_ctx* ctx) { return ctx ? ctx->B.NJ : ARMOUR_ERR_ARG; }
int armour_num_time_steps(const armour_ctx* ctx) { return ctx ? ctx->B.T : ARMOUR_ERR_ARG; }
int armour_num_constraints(const armour_ctx* ctx, int nobs) {
    if (!ctx || nobs < 0) return ARMOUR_ERR_ARG;
    return NF * ctx->B.T + ctx->B.NJ * ctx->B.T * nobs + 4 * NF;
}

int armour_ctx_reserve(armour_ctx* ctx, int nprob, int nobs) {
    int rc = check_batch(ctx, nprob, nobs);
    if (rc) return rc;
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    rc = ensure_obstacle_buffers(ctx, nprob, nobs);  // (reserving does not change the current batch)
    if (rc) return rc;
    return ensure_eval_buffers(ctx, size_t(nprob) * armour_num_constraints(ctx, nobs), true, true);
}

// ---- build -----------------------------------------------------------------------------------------
int armour_batch_reachsets_build_device(armour_ctx* ctx, int nprob, const double* d_q0, const double* d_qd0,
                                        const double* d_qdd0, const double* d_obstacles, int nobs) {
    int rc = check_batch(ctx, nprob, nobs);
    if (rc) return rc;
    if (!d_q0 || !d_qd0 || !d_qdd0 || (nobs > 0 && !d_obstacles)) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    rc = ensure_obstacle_buffers(ctx, nprob, nobs);
    if (rc) return rc;
    ctx->B.O = nobs;
    ctx->B.nprob = nprob;
    double* d_in = ctx->d_in.get();
    const size_t P = size_t(ctx->cfg.max_problems);
    ctx->B.epoch++;
    int nl = 0;
    bool latency = false;
    if (nobs > 0) {
        // the kernels read the caller's buffers; k_hyperplanes copies them into the context's own (for the evaluations that
        // follow) — no copies in front of the build.  In the latency configuration k_hyperplanes is a programmatic dependent
        // of k_reachsets and starts on the intervals that are complete.
        Batch Bb = ctx->B;
        Bb.q0 = d_q0;
        Bb.qd0 = d_qd0;
        Bb.qdd0 = d_qdd0;
        Bb.obstacles = d_obstacles;
        { int rc2 = launch_build(ctx, Bb, &nl, &latency); if (rc2) return rc2; }
        HpStage stage{d_in, d_in + P * NF, d_in + 2 * P * NF, ctx->d_obs.get()};
        CU(launch_hyperplanes(Bb, ctx->stream, latency ? ctx->d_unit_flag.get() : nullptr, stage));
        nl++;
    } else {
        const size_t nb = size_t(nprob) * NF * sizeof(double);
        CU(cudaMemcpyAsync(d_in, d_q0, nb, cudaMemcpyDeviceToDevice, ctx->stream));
        CU(cudaMemcpyAsync(d_in + P * NF, d_qd0, nb, cudaMemcpyDeviceToDevice, ctx->stream));
        CU(cudaMemcpyAsync(d_in + 2 * P * NF, d_qdd0, nb, cudaMemcpyDeviceToDevice, ctx->stream));
        { int rc2 = launch_build(ctx, ctx->B, &nl, &latency); if (rc2) return rc2; }
    }
    CU(launch_pack_image(ctx->B, ctx->stream));
    nl++;
    ctx->launches += nl;
    ctx->built_nprob = nprob;
    ctx->h_torque_valid = false;
    ctx->h_q0.clear();
    return ARMOUR_OK;
}

int armour_batch_reachsets_build(armour_ctx* ctx, int nprob, const double* q0, const double* qd0, const double* qdd0,
                                 const double* obstacles, int nobs) {
    int rc = check_batch(ctx, nprob, nobs);
    if (rc) return rc;
    if (!q0 || !qd0 || !qdd0 || (nobs > 0 && !obstacles)) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    rc = ensure_obstacle_buffers(ctx, nprob, nobs);
    if (rc) return rc;
    ctx->B.O = nobs;
    ctx->B.nprob = nprob;
    double* d_in = ctx->d_in.get();
    const size_t P = size_t(ctx->cfg.max_problems);
    const size_t nb = size_t(nprob) * NF * sizeof(double);
    CU(cudaMemcpyAsync(d_in, q0, nb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_in + P * NF, qd0, nb, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d_in + 2 * P * NF, qdd0, nb, cudaMemcpyHostToDevice, ctx->stream));
    if (nobs > 0)
        CU(cudaMemcpyAsync(ctx->d_obs.get(), obstacles, size_t(nprob) * nobs * 12 * sizeof(double), cudaMemcpyHostToDevice,
                           ctx->stream));
    ctx->B.epoch++;
    int nl = 0;
    bool latency = false;
    { int rc2 = launch_build(ctx, ctx->B, &nl, &latency); if (rc2) return rc2; }
    ctx->launches += nl;
    CU(launch_hyperplanes(ctx->B, ctx->stream, (latency && nobs > 0) ? ctx->d_unit_flag.get() : nullptr));
    ctx->launches += (nobs > 0);
    CU(launch_pack_image(ctx->B, ctx->stream));
    ctx->launches++;
    ctx->built_nprob = nprob;
    ctx->h_torque_valid = false;
    ctx->h_q0.assign(q0, q0 + size_t(nprob) * NF);
    ctx->h_qd0.assign(qd0, qd0 + size_t(nprob) * NF);
    ctx->h_qdd0.assign(qdd0, qdd0 + size_t(nprob) * NF);
    // surface capacity overflows of the build (never truncate silently)
    std::vector<int> st(nprob);
    CU(cudaMemcpyAsync(st.data(), ctx->B.status, nprob * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    for (int p = 0; p < nprob; p++)
        if ((st[p] >> 3) == ctx->B.epoch && (st[p] & 7) != 0) {
            // which check failed first, and where (diagnostics of the build kernel: stats[4..6])
            int site[3] = {0, 0, 0};
            const int* dstats = latency ? ctx->k1_lat.stats : ctx->k1_thr.stats;
            std::string where;
            if (dstats && cudaMemcpy(site, dstats + 4, sizeof(site), cudaMemcpyDeviceToHost) == cudaSuccess && site[2] == ctx->B.epoch) {
                const int line = site[0] >> 3;
                where = "; first failing check: code " + std::to_string(site[0] & 7) + " at " +
                        (line >= 10000 ? "k1_reachsets.cuh:" + std::to_string(line - 10000) : "k1_pz.cuh:" + std::to_string(line)) +
                        ", problem " + std::to_string(site[1] / ctx->B.T) + " interval " + std::to_string(site[1] % ctx->B.T);
            }
            return fail(ctx, ARMOUR_ERR_CAPACITY,
                        "reach-set build overflowed a monomial table (problem " + std::to_string(p) + ", code " +
                            std::to_string(st[p] & 7) + ")" + where);
        }
    return ARMOUR_OK;
}

int armour_reachsets_build(armour_ctx* ctx, const double* q0, const double* qd0, const double* qdd0,
                           const double* obstacles, int nobs) {
    return armour_batch_reachsets_build(ctx, 1, q0, qd0, qdd0, obstacles, nobs);
}

int armour_batch_get_build_status(armour_ctx* ctx, int nprob, int* out) {
    if (!ctx || !out || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    CU(cudaMemcpyAsync(out, ctx->B.status, nprob * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    for (int p = 0; p < nprob; p++)  // device words are stamped with the build ordinal: report this build's code only
        out[p] = ((out[p] >> 3) == ctx->B.epoch && (out[p] & 7) != 0) ? ARMOUR_ERR_CAPACITY : ARMOUR_OK;
    return ARMOUR_OK;
}

int armour_batch_get_monomial_counts(armour_ctx* ctx, int nprob, int* link_n, int* u_n) {
    if (!ctx || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    const size_t T = ctx->B.T, NJ = ctx->B.NJ;
    if (link_n)
        CU(cudaMemcpyAsync(link_n, ctx->B.link_n, nprob * T * NJ * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (u_n) CU(cudaMemcpyAsync(u_n, ctx->B.u_n, nprob * T * NF * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

int armour_batch_get_candidate_counts(armour_ctx* ctx, int nprob, unsigned char* out) {
    if (!ctx || !out || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    const size_t rows = size_t(ctx->B.NJ) * ctx->B.T * ctx->B.O;
    if (rows) CU(cudaMemcpyAsync(out, ctx->B.hp_cnt, nprob * rows, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

int armour_chunk_intervals(void) { return TB; }

int armour_eval_image_layout(armour_ctx* ctx, long long* layout) {
    if (!ctx || !layout) return ARMOUR_ERR_ARG;
    const Batch& B = ctx->B;
    const size_t v[10] = {B.img_chunk(), 0, B.img_ut(), B.img_lc(), B.img_lr(), B.img_uc(), B.img_ur(), B.img_grp(), B.img_cnt(), B.img_hdr()};
    for (int i = 0; i < 10; i++) layout[i] = (long long)v[i];
    return ARMOUR_OK;
}

int armour_batch_get_eval_images(armour_ctx* ctx, int nprob, void* out) {
    if (!ctx || !out || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    CU(cudaMemcpyAsync(out, ctx->B.img, size_t(nprob) * (ctx->B.T / TB) * ctx->B.img_chunk(), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

#ifdef K1_PROFILE
// developer builds only: per-(interval, operation site) cycle counts of the last single-problem builds
extern "C" int armour_debug_k1_profile(long long* out, int reset) {
    cudaDeviceSynchronize();
    if (out) {
        int sp[8];
        if (cudaMemcpyFromSymbol(sp, g_k1spill, sizeof(sp)) == cudaSuccess)
            std::printf("k1 profile: %d of %d arena blocks in global memory, %d scratch pools in global memory, %d cross products on "
                        "the table path (largest term count %d)\n", sp[0], sp[1], sp[2], sp[3], sp[4]);
    }
    if (out && cudaMemcpyFromSymbol(out, g_k1prof, sizeof(long long) * 128 * K1_PROF_SITES * 2) != cudaSuccess) return ARMOUR_ERR_CUDA;
    if (reset) {
        void* p = nullptr;
        if (cudaGetSymbolAddress(&p, g_k1prof) != cudaSuccess) return ARMOUR_ERR_CUDA;
        if (cudaMemset(p, 0, sizeof(long long) * 128 * K1_PROF_SITES * 2) != cudaSuccess) return ARMOUR_ERR_CUDA;
    }
    return ARMOUR_OK;
}
#endif

int armour_measure_fp64_peak(armour_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return ARMOUR_ERR_ARG;
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->cfg.device));
    DeviceBuffer<double> d_out;
    CU(d_out.reserve(1));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    const int iters = 4096, grid = sms * 8, block = 256;
    double best = 0.0;
    auto run = [&]() -> int {
        CU(cudaEventCreate(&e0));
        CU(cudaEventCreate(&e1));
        for (int rep = 0; rep < 4; rep++) {
            CU(cudaEventRecord(e0, ctx->stream));
            k_fp64_peak<<<grid, block, 0, ctx->stream>>>(d_out.get(), iters, 1.0000001);
            CU(cudaEventRecord(e1, ctx->stream));
            CU(cudaEventSynchronize(e1));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, e0, e1));
            const double fl = 2.0 * 8 * double(iters) * double(grid) * block;
            if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
        }
        ctx->launches += 4;
        return ARMOUR_OK;
    };
    const int rc = run();
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (rc == ARMOUR_OK) *tflops = best;
    return rc;
}

// ---- evaluate --------------------------------------------------------------------------------------
int armour_batch_eval_device(armour_ctx* ctx, int nprob, const double* d_k, double* d_g, double* d_values) {
    if (!ctx || !d_k) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "evaluate before build");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    Batch B = ctx->B;
    B.nprob = nprob;
    CU(launch_constraints(B, d_k, d_g, d_values, ctx->stream));
    ctx->launches += 1 + (B.O > 0);
    return ARMOUR_OK;
}

int armour_batch_eval(armour_ctx* ctx, int nprob, const double* k, double* g, double* values) {
    if (!ctx || !k) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "evaluate before build");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    const size_t m = size_t(ctx->B.m());
    int rc = ensure_eval_buffers(ctx, nprob * m, g != nullptr, values != nullptr);
    if (rc) return rc;
    CU(cudaMemcpyAsync(ctx->d_k.get(), k, size_t(nprob) * NF * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    rc = armour_batch_eval_device(ctx, nprob, ctx->d_k.get(), g ? ctx->d_g.get() : nullptr, values ? ctx->d_jac.get() : nullptr);
    if (rc) return rc;
    if (g) CU(cudaMemcpyAsync(g, ctx->d_g.get(), nprob * m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (values)
        CU(cudaMemcpyAsync(values, ctx->d_jac.get(), nprob * m * NF * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

// ---- structured Jacobian (offered beside the dense one; the reference declares its Jacobian dense) ------------------
long long armour_jacobian_nnz(const armour_ctx* ctx, int nobs) {
    if (!ctx || nobs < 0) return ARMOUR_ERR_ARG;
    return jac_nnz(ctx->B.T, ctx->B.NJ, nobs);
}

int armour_jacobian_structure(const armour_ctx* ctx, int nobs, int* iRow, int* jCol) {
    if (!ctx || nobs < 0 || !iRow || !jCol) return ARMOUR_ERR_ARG;
    const int T = ctx->B.T, NJ = ctx->B.NJ;
    size_t n = 0;
    for (int r = 0; r < NF * T; r++)
        for (int c = 0; c < NF; c++, n++) {
            iRow[n] = r;
            jCol[n] = c;
        }
    for (int l = 0; l < NJ; l++)
        for (int r = 0; r < T * nobs; r++)
            for (int c = 0; c < jac_link_width(l); c++, n++) {
                iRow[n] = NF * T + l * T * nobs + r;
                jCol[n] = c;
            }
    for (int r = 0; r < 4 * NF; r++, n++) {
        iRow[n] = NF * T + NJ * T * nobs + r;
        jCol[n] = r % NF;
    }
    return ARMOUR_OK;
}

int armour_batch_eval_structured_device(armour_ctx* ctx, int nprob, const double* d_k, double* d_g, double* d_values_nnz) {
    if (!ctx || !d_k || !d_values_nnz) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "evaluate before build");
    CU(cudaSetDevice(ctx->cfg.device));
    int rc = ensure_eval_buffers(ctx, size_t(nprob) * ctx->B.m(), false, true);
    if (rc) return rc;
    rc = armour_batch_eval_device(ctx, nprob, d_k, d_g, ctx->d_jac.get());
    if (rc) return rc;
    Batch B = ctx->B;
    B.nprob = nprob;
    CU(launch_pack_jacobian(B, ctx->d_jac.get(), d_values_nnz, ctx->stream));
    ctx->launches += 1;
    return ARMOUR_OK;
}

int armour_batch_eval_structured(armour_ctx* ctx, int nprob, const double* k, double* g, double* values_nnz) {
    if (!ctx || !k || !values_nnz) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "evaluate before build");
    CU(cudaSetDevice(ctx->cfg.device));
    const size_t m = size_t(ctx->B.m());
    int rc = ensure_eval_buffers(ctx, nprob * m, g != nullptr, true);
    if (rc) return rc;
    const size_t nnz = size_t(jac_nnz(ctx->B.T, ctx->B.NJ, ctx->B.O));
    CU(ctx->d_jnz.reserve(nprob * nnz));
    CU(cudaMemcpyAsync(ctx->d_k.get(), k, size_t(nprob) * NF * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    rc = armour_batch_eval_structured_device(ctx, nprob, ctx->d_k.get(), g ? ctx->d_g.get() : nullptr, ctx->d_jnz.get());
    if (rc) return rc;
    if (g) CU(cudaMemcpyAsync(g, ctx->d_g.get(), nprob * m * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(values_nnz, ctx->d_jnz.get(), nprob * nnz * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

int armour_eval_jac_g_structured(armour_ctx* ctx, const double* k, double* values_nnz) {
    return armour_batch_eval_structured(ctx, 1, k, nullptr, values_nnz);
}

int armour_eval_g(armour_ctx* ctx, const double* k, double* g) { return armour_batch_eval(ctx, 1, k, g, nullptr); }
int armour_eval_jac_g(armour_ctx* ctx, const double* k, double* values) {
    return armour_batch_eval(ctx, 1, k, nullptr, values);
}
int armour_eval_g_jac(armour_ctx* ctx, const double* k, double* g, double* values) {
    return armour_batch_eval(ctx, 1, k, g, values);
}

int armour_batch_verdict_device(armour_ctx* ctx, int nprob, const double* d_g, int* d_feasible, int* d_first) {
    if (!ctx || !d_g || !d_feasible || !d_first) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "verdict before build");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    Batch B = ctx->B;
    B.nprob = nprob;
    CU(launch_verdict(B, d_g, d_feasible, d_first, ctx->stream));
    ctx->launches += 1;
    return ARMOUR_OK;
}

// ---- batched device solver (SURVEY 8f-1) -------------------------------------------------------------
void armour_solver_options_default(armour_solver_options* opt) {
    if (!opt) return;
    opt->max_iter = 60;
    opt->tol = 1e-4;
    opt->torque_tol = 1e-2;
    opt->collision_tol = 1e-4;
    opt->qp_sweeps = 200;
    opt->qp_update_budget = 16384;
}

}  // extern "C"

namespace {

// The batched solver's host loop over one NLP policy (csrc/k4_solver.cuh).  eval(Bb, x, g, jac) is one evaluation step of the
// problems of Bb at x into the policy's row layout (jac may be nullptr) and launches n_eval kernels; verdict(g, feasible, first)
// is the final verdict of the whole batch.  g_x / jac_x: [nprob][m] / [nprob][m][NF] buffers of the evaluation at the iterate.
template <class Nlp, class Eval, class Verdict>
int run_solver(armour_ctx* ctx, int nprob, const double* d_q_des, const armour_solver_options& opt, const Nlp& nlp, int m_rows,
               double* g_x, double* jac_x, const Eval& eval, int n_eval, const Verdict& verdict, double* d_k_opt, int* d_feasible,
               int* d_first, int* d_iters) {
    if (opt.max_iter < 1 || !(opt.tol > 0) || opt.qp_sweeps < 1) return fail(ctx, ARMOUR_ERR_ARG, "solver options");
    Batch B = ctx->B;
    B.nprob = nprob;
    const size_t m = size_t(m_rows);
    // scratch: state arrays + second g buffer + linearised rows.  Its size depends on nprob AND on m (obstacle count of
    // the current batch): capacity is tracked in elements and the layout below always uses this call's nprob.
    const size_t P = size_t(nprob);
    CU(ctx->d_solver.reserve(P * (3 * NF + 4) + P * m + P * SOLVER_ROWCAP * SOLVER_ROWW));
    CU(ctx->d_solver_i.reserve(8 * P + 1));
    SolverState S;
    double* w = ctx->d_solver.get();
    S.x = w; w += P * NF;
    S.xt = w; w += P * NF;
    S.best = w; w += P * NF;
    S.f = w; w += P;
    S.viol = w; w += P;
    S.fbest = w; w += P;
    S.delta = w; w += P;
    double* d_gt = w; w += P * m;
    S.rows = w;
    S.have_best = ctx->d_solver_i.get();
    S.status = S.have_best + P;
    S.iters = S.status + P;
    S.evals = S.iters + P;
    S.dbg = S.evals + P;
    int* d_running = S.dbg + 3 * P;
    int* d_list = d_running + 1;  // [P] problems still running
    S.q_des = d_q_des;
    S.tol = opt.tol;
    S.torque_tol = opt.torque_tol;
    S.collision_tol = opt.collision_tol;
    S.max_iter = opt.max_iter;
    S.qp_sweeps = opt.qp_sweeps;
    S.qp_update_budget = opt.qp_update_budget;
    cudaStream_t st = ctx->stream;
    const size_t step_smem = solver_step_smem(m_rows);  // ballot masks of the row gathering: 64 B per 256 rows
    if (step_smem > 200 * 1024) return fail(ctx, ARMOUR_ERR_ARG, "too many constraint rows for the batched solver");
    if (step_smem > 40 * 1024)  // beyond the default limit (a few hundred obstacles): opt in, per device (cheap, idempotent)
        CU(cudaFuncSetAttribute(k_solver_step<Nlp>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(step_smem)));
    // x = 0 (armtd_NLP::get_starting_point), g(0)
    CU(cudaMemsetAsync(S.x, 0, size_t(nprob) * NF * sizeof(double), st));
    CU(cudaMemsetAsync(S.xt, 0, size_t(nprob) * NF * sizeof(double), st));
    { int rc = eval(B, S.x, g_x, nullptr); if (rc) return rc; }
    k_solver_start<<<nprob, SOLVER_THREADS, 0, st>>>(B, nlp, S, g_x);
    CU(cudaGetLastError());
    ctx->launches += 1 + n_eval;
    // the list of running problems is rebuilt every `compact_every` iterations (a host synchronisation each time; between two
    // rebuilds the solver kernels skip finished problems themselves, only the constraint kernel still evaluates them)
    static const int compact_every = [] {
        const char* v = std::getenv("ARMOUR_SOLVER_COMPACT_EVERY");  // developer knob
        const int n = v ? std::atoi(v) : 0;
        return n >= 1 ? n : 4;
    }();
    Batch Ba = B;      // launches over the problems still running (all of them at first)
    int nactive = nprob;
    for (int it = 0; it < opt.max_iter && nactive > 0; it++) {
        Ba.nprob = nactive;
        { int rc = eval(Ba, S.x, g_x, jac_x); if (rc) return rc; }
        k_solver_step<<<nactive, SOLVER_THREADS, step_smem, st>>>(Ba, nlp, S, g_x, jac_x, it);
        { int rc = eval(Ba, S.xt, d_gt, nullptr); if (rc) return rc; }
        k_solver_accept<<<nactive, SOLVER_THREADS, 0, st>>>(Ba, nlp, S, d_gt, it == opt.max_iter - 1 ? 1 : 0);
        CU(cudaGetLastError());  // (covers k_solver_step too: launch errors are sticky until read)
        ctx->launches += 2 + 2 * n_eval;
        if ((it + 1) % compact_every == 0 && it + 1 < opt.max_iter) {  // every fourth iteration: who is still running?
            CU(cudaMemsetAsync(d_running, 0, sizeof(int), st));
            k_solver_compact<<<(nprob + 255) / 256, 256, 0, st>>>(S, nprob, d_running, d_list);
            CU(cudaMemcpyAsync(&nactive, d_running, sizeof(int), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            ctx->launches += 1;
            Ba.plist = d_list;
        }
    }
    k_solver_final<<<(nprob + 255) / 256, 256, 0, st>>>(S, nprob, d_k_opt, nullptr);
    { int rc = eval(B, d_k_opt, g_x, nullptr); if (rc) return rc; }
    { int rc = verdict(g_x, d_feasible, d_first); if (rc) return rc; }
    if (d_iters) CU(cudaMemcpyAsync(d_iters, S.iters, size_t(nprob) * sizeof(int), cudaMemcpyDeviceToDevice, st));
    if (std::getenv("ARMOUR_SOLVER_DEBUG")) {  // developer aid: row / active-set iteration / drop counts of the last step per problem
        std::vector<int> dbg(size_t(nprob) * 3);
        CU(cudaMemcpyAsync(dbg.data(), S.dbg, dbg.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        long long r = 0, sw = 0, mv = 0;
        int rmax = 0, mvmax = 0;
        for (int p = 0; p < nprob; p++) {
            r += dbg[p * 3];
            sw += dbg[p * 3 + 1];
            mv += dbg[p * 3 + 2];
            rmax = std::max(rmax, dbg[p * 3]);
            mvmax = std::max(mvmax, dbg[p * 3 + 2]);
        }
        std::printf("solver debug: last step per problem: rows mean %.0f max %d, active-set iterations mean %.1f, dropped rows mean %.1f max %d\n",
                    double(r) / nprob, rmax, double(sw) / nprob, double(mv) / nprob, mvmax);
    }
    ctx->launches += 2 + n_eval;  // k_solver_final, the evaluation at k_opt, the verdict
    CU(cudaGetLastError());
    return ARMOUR_OK;
}

// host-pointer front of a *_solve_device call: stages q_des in, k_opt and the verdicts out
using SolveDeviceFn = int (*)(armour_ctx*, int, const double*, const armour_solver_options*, double*, int*, int*, int*);
int solve_from_host(armour_ctx* ctx, int nprob, const double* q_des, const armour_solver_options* opt, double* k_opt, int* feasible,
                    int* first_violation, int* iterations, SolveDeviceFn solve_device) {
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    const size_t nk = size_t(nprob) * NF * sizeof(double), ni = size_t(nprob) * sizeof(int);
    void* d[5];  // q_des, k_opt, feasible, first violation, iterations
    int rc = stage(ctx, {nk, nk, ni, ni, ni}, d);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(d[0], q_des, nk, cudaMemcpyHostToDevice, st));
    rc = solve_device(ctx, nprob, static_cast<double*>(d[0]), opt, static_cast<double*>(d[1]), static_cast<int*>(d[2]),
                      static_cast<int*>(d[3]), static_cast<int*>(d[4]));
    if (rc) return rc;
    CU(cudaMemcpyAsync(k_opt, d[1], nk, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(feasible, d[2], ni, cudaMemcpyDeviceToHost, st));
    if (first_violation) CU(cudaMemcpyAsync(first_violation, d[3], ni, cudaMemcpyDeviceToHost, st));
    if (iterations) CU(cudaMemcpyAsync(iterations, d[4], ni, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}

}  // namespace

extern "C" {

int armour_batch_solve_device(armour_ctx* ctx, int nprob, const double* d_q_des, const armour_solver_options* opt_in,
                              double* d_k_opt, int* d_feasible, int* d_first, int* d_iters) {
    if (!ctx || !d_q_des || !d_k_opt || !d_feasible || !d_first) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "solve before build");
    armour_solver_options opt;
    armour_solver_options_default(&opt);
    if (opt_in) opt = *opt_in;
    if (opt.max_iter < 1 || !(opt.tol > 0) || opt.qp_sweeps < 1) return fail(ctx, ARMOUR_ERR_ARG, "solver options");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    int rc = ensure_eval_buffers(ctx, size_t(nprob) * ctx->B.m(), true, true);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    auto eval = [ctx, st](const Batch& Bb, const double* x, double* g, double* jac) {
        CU(launch_constraints(Bb, x, g, jac, st));
        return int(ARMOUR_OK);
    };
    auto verdict = [ctx, st, nprob](const double* g, int* feasible, int* first) {
        Batch B = ctx->B;
        B.nprob = nprob;
        CU(launch_verdict(B, g, feasible, first, st));
        return int(ARMOUR_OK);
    };
    return run_solver(ctx, nprob, d_q_des, opt, ArmourNlp{}, ctx->B.m(), ctx->d_g.get(), ctx->d_jac.get(), eval, 1 + (ctx->B.O > 0),
                      verdict, d_k_opt, d_feasible, d_first, d_iters);
}

int armour_batch_solve(armour_ctx* ctx, int nprob, const double* q_des, const armour_solver_options* opt, double* k_opt,
                       int* feasible, int* first_violation, int* iterations) {
    if (!ctx || !q_des || !k_opt || !feasible) return ARMOUR_ERR_ARG;
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, "solve before build");
    return solve_from_host(ctx, nprob, q_des, opt, k_opt, feasible, first_violation, iterations, armour_batch_solve_device);
}

void armour_rollout_options_default(armour_rollout_options* opt) {
    if (!opt) return;
    std::memset(opt, 0, sizeof(*opt));
    opt->struct_size = int(sizeof(armour_rollout_options));
    opt->max_replans = 100;
    opt->lookahead = 0.1;
    opt->goal_radius = 0.05;
    opt->audit_samples = 16;
    armour_solver_options_default(&opt->solver);
}

}  // extern "C"

namespace {

// armtd: the call runs episodes of the ARMTD comparison planner (armour_armtd_batch_rollout*), which need a context of that planner
int check_rollout(armour_ctx* ctx, int nworlds, int nobs, const armour_rollout_options* opt, bool armtd) {
    if (!ctx) return ARMOUR_ERR_ARG;
    if (ctx->armtd && !armtd)
        return fail(ctx, ARMOUR_ERR_STATE, "armour_batch_rollout runs the main planner: use armour_armtd_batch_rollout on an ARMTD context");
    if (!ctx->armtd && armtd)
        return fail(ctx, ARMOUR_ERR_STATE, "not an ARMTD context (armour_armtd_ctx_create / armour_armtd_batch_ctx_create)");
    if (nworlds < 1) return fail(ctx, ARMOUR_ERR_ARG, "nworlds < 1");
    if (nworlds > ctx->cfg.max_problems) return fail(ctx, ARMOUR_ERR_STATE, "nworlds larger than max_problems");
    if (nobs < 0) return fail(ctx, ARMOUR_ERR_ARG, "negative obstacle count");
    if (nobs > ctx->cfg.max_obstacles) return fail(ctx, ARMOUR_ERR_OBSTACLES, "number of obstacles larger than max_obstacles");
    if (!opt || opt->struct_size != int(sizeof(armour_rollout_options))) return fail(ctx, ARMOUR_ERR_ARG, "rollout options");
    if (opt->max_replans < 1 || opt->audit_samples < 2 || !(opt->lookahead > 0) || !(opt->goal_radius >= 0))
        return fail(ctx, ARMOUR_ERR_ARG, "rollout options");
    const armour_solver_options& so = opt->solver;
    if (so.max_iter < 1 || !(so.tol > 0) || so.qp_sweeps < 1 || !(so.collision_tol >= 0))
        return fail(ctx, ARMOUR_ERR_ARG, "solver options");
    return ARMOUR_OK;
}

// The planner policies of the episode loop.  extra: doubles of rollout scratch per world beyond the common arrays, bound by
// bind(w, N); plan(): the build and solve of the dense batch of nrun running worlds into D.dk / dfeas / dfirst / diters;
// traj(): the trajectory class of k_rollout_advance.
// The main planner: armour_batch_reachsets_build_device + armour_batch_solve_device, the Bezier of its plans.
struct ArmourEpisodes {
    static constexpr size_t extra = 0;
    void bind(double*, size_t) {}
    int plan(armour_ctx* ctx, const RolloutDev& D, int nrun, int nobs, const armour_solver_options& so) const {
        int rc = armour_batch_reachsets_build_device(ctx, nrun, D.dq0, D.dqd0, D.dqdd0, nobs > 0 ? D.dobs : nullptr, nobs);
        if (rc) return rc;
        return armour_batch_solve_device(ctx, nrun, D.dq_des, &so, D.dk, D.dfeas, D.dfirst, D.diters);
    }
    RollBezier traj() const { return {}; }
};
// The ARMTD comparison planner: a prepare step (k_armtd_offline_jrs deriving k_range from qd0 and the stand-in table of every
// running world), armour_armtd_batch_build_device with the device's sincos + armour_armtd_batch_solve_device, the
// constant-acceleration curve.  Scratch: k_range [N][NF] and the table [N][6][NF][100] of the dense batch.
struct ArmtdEpisodes {
    static constexpr size_t extra = NF + 6 * NF * ARMTD_T;
    double* k_range = nullptr;
    double* jrs = nullptr;
    void bind(double* w, size_t N) {
        k_range = w;
        jrs = w + N * NF;
    }
    int plan(armour_ctx* ctx, const RolloutDev& D, int nrun, int nobs, const armour_solver_options& so) const {
        CU(launch_armtd_offline_jrs(nrun, D.dqd0, nullptr, k_range, jrs, ctx->stream));
        ctx->launches += 1;
        int rc = armour_armtd_batch_build_device(ctx, nrun, D.dq0, D.dqd0, jrs, k_range, nobs > 0 ? D.dobs : nullptr, nobs, nullptr);
        if (rc) return rc;
        return armour_armtd_batch_solve_device(ctx, nrun, D.dq_des, &so, D.dk, D.dfeas, D.dfirst, D.diters);
    }
    RollConstAcc traj() const { return {k_range}; }
};

// The episode loop (include/armour_b200.h, "closed-loop replanning episodes"): per replan k_rollout_plan, the planner's device
// build and solve of the running worlds, k_rollout_advance, k_clearance over the audit samples, k_rollout_finish; then one copy
// of the running count to the host and one synchronisation.
template <class Episodes>
int rollout_run(armour_ctx* ctx, int n, const double* d_start, const double* d_goal, const double* d_obstacles, int nobs,
                const armour_rollout_options& opt, const armour_rollout_out& out) {
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    const size_t N = size_t(n), S = size_t(opt.audit_samples), no = size_t(nobs) * 12;
    CU(ctx->d_roll.reserve(N * (ROLL_STATE + ROLL_PLAN + 1 + 5 * NF + 1) + N * no + N * S * NF + N * Episodes::extra));
    Episodes ep;
    CU(ctx->d_roll_i.reserve(10 * N + 1));
    RolloutDev D;
    D.n = n;
    D.R = opt.max_replans;
    D.nobs = nobs;
    D.S = opt.audit_samples;
    D.lookahead = opt.lookahead;
    D.goal_radius = opt.goal_radius;
    D.collision_tol = opt.solver.collision_tol;
    D.start = d_start;
    D.goal = d_goal;
    D.obstacles = d_obstacles;
    double* w = ctx->d_roll.get();
    D.state = w; w += N * ROLL_STATE;
    D.plan = w; w += N * ROLL_PLAN;
    D.minc = w; w += N;
    D.dq0 = w; w += N * NF;
    D.dqd0 = w; w += N * NF;
    D.dqdd0 = w; w += N * NF;
    D.dq_des = w; w += N * NF;
    D.dk = w; w += N * NF;
    D.dclear = w; w += N;
    D.dobs = w; w += N * no;
    D.samp = w; w += N * S * NF;
    ep.bind(w, N);
    int* wi = ctx->d_roll_i.get();
    D.outcome = wi; wi += N;
    D.replans = wi; wi += N;
    D.infeasible = wi; wi += N;
    D.limit = wi; wi += N;
    D.dfeas = wi; wi += N;
    D.dfirst = wi; wi += N;
    D.diters = wi; wi += N;
    int* list = wi; wi += N;
    int* next = wi; wi += N;
    int* d_count = wi;
    D.log_state = out.log_state;
    D.log_q_des = out.log_q_des;
    D.log_k = out.log_k;
    D.log_int = out.log_int;
    D.log_clearance = out.log_clearance;
    cudaStream_t st = ctx->stream;
    const int ib = std::min<int>(int((N * size_t(opt.max_replans) + ROLL_THREADS - 1) / ROLL_THREADS), 4096);
    k_rollout_init<<<ib, ROLL_THREADS, 0, st>>>(D, list);
    CU(cudaGetLastError());
    ctx->launches += 1;
    int nrun = n;
    for (int r = 0; r < opt.max_replans && nrun > 0; r++) {
        const int gb = (nrun + ROLL_THREADS - 1) / ROLL_THREADS;
        k_rollout_plan<<<gb, ROLL_THREADS, 0, st>>>(D, r, nrun, list);
        CU(cudaGetLastError());
        ctx->launches += 1;
        { int rc = ep.plan(ctx, D, nrun, nobs, opt.solver); if (rc) return rc; }
        k_rollout_advance<<<gb, ROLL_THREADS, 0, st>>>(D, r, nrun, list, ctx->B.status, ctx->B.epoch, ep.traj());
        k_clearance<<<nrun, CLEAR_THREADS, 0, st>>>(D.samp, opt.audit_samples, list, d_obstacles, nobs, D.dclear, nullptr);
        k_rollout_finish<<<1, FINISH_THREADS, 0, st>>>(D, r, nrun, list, next, d_count);
        CU(cudaGetLastError());
        ctx->launches += 3;
        CU(cudaMemcpyAsync(&nrun, d_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        std::swap(list, next);
    }
    if (out.outcome) CU(cudaMemcpyAsync(out.outcome, D.outcome, N * sizeof(int), cudaMemcpyDeviceToDevice, st));
    if (out.replans) CU(cudaMemcpyAsync(out.replans, D.replans, N * sizeof(int), cudaMemcpyDeviceToDevice, st));
    if (out.infeasible) CU(cudaMemcpyAsync(out.infeasible, D.infeasible, N * sizeof(int), cudaMemcpyDeviceToDevice, st));
    if (out.final_state) CU(cudaMemcpyAsync(out.final_state, D.state, N * ROLL_STATE * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (out.min_clearance) CU(cudaMemcpyAsync(out.min_clearance, D.minc, N * sizeof(double), cudaMemcpyDeviceToDevice, st));
    return ARMOUR_OK;
}

int run_episodes(armour_ctx* ctx, bool armtd, int n, const double* d_start, const double* d_goal, const double* d_obstacles, int nobs,
                 const armour_rollout_options& opt, const armour_rollout_out& out) {
    if (armtd) return rollout_run<ArmtdEpisodes>(ctx, n, d_start, d_goal, d_obstacles, nobs, opt, out);
    return rollout_run<ArmourEpisodes>(ctx, n, d_start, d_goal, d_obstacles, nobs, opt, out);
}

int rollout_device(armour_ctx* ctx, int nworlds, const double* d_start, const double* d_goal, const double* d_obstacles, int nobs,
                   const armour_rollout_options* opt, const armour_rollout_out* d_out, bool armtd) {
    int rc = check_rollout(ctx, nworlds, nobs, opt, armtd);
    if (rc) return rc;
    if (!d_start || !d_goal || (nobs > 0 && !d_obstacles) || !d_out) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    return run_episodes(ctx, armtd, nworlds, d_start, d_goal, d_obstacles, nobs, *opt, *d_out);
}

// host-pointer front of the episodes: stages the inputs in and the requested outputs out
int rollout_host(armour_ctx* ctx, int nworlds, const double* start, const double* goal, const double* obstacles, int nobs,
                 const armour_rollout_options* opt, const armour_rollout_out* out, bool armtd) {
    int rc = check_rollout(ctx, nworlds, nobs, opt, armtd);
    if (rc) return rc;
    if (!start || !goal || (nobs > 0 && !obstacles) || !out) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    CU(cudaSetDevice(ctx->cfg.device));
    const size_t N = size_t(nworlds), R = size_t(opt->max_replans);
    // inputs, then one device array per requested output
    const size_t sz[13] = {N * NF * 8, N * NF * 8, N * size_t(nobs) * 12 * 8,
                           out->outcome ? N * 4 : 0, out->replans ? N * 4 : 0, out->infeasible ? N * 4 : 0,
                           out->final_state ? N * ROLL_STATE * 8 : 0, out->min_clearance ? N * 8 : 0,
                           out->log_state ? R * N * ROLL_STATE * 8 : 0, out->log_q_des ? R * N * NF * 8 : 0,
                           out->log_k ? R * N * NF * 8 : 0, out->log_int ? R * N * 4 * 4 : 0, out->log_clearance ? R * N * 8 : 0};
    void* d[13];
    rc = stage(ctx, sz, d);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(d[0], start, sz[0], cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d[1], goal, sz[1], cudaMemcpyHostToDevice, st));
    if (nobs > 0) CU(cudaMemcpyAsync(d[2], obstacles, sz[2], cudaMemcpyHostToDevice, st));
    armour_rollout_out d_out;
    d_out.outcome = static_cast<int*>(d[3]);
    d_out.replans = static_cast<int*>(d[4]);
    d_out.infeasible = static_cast<int*>(d[5]);
    d_out.final_state = static_cast<double*>(d[6]);
    d_out.min_clearance = static_cast<double*>(d[7]);
    d_out.log_state = static_cast<double*>(d[8]);
    d_out.log_q_des = static_cast<double*>(d[9]);
    d_out.log_k = static_cast<double*>(d[10]);
    d_out.log_int = static_cast<int*>(d[11]);
    d_out.log_clearance = static_cast<double*>(d[12]);
    rc = run_episodes(ctx, armtd, nworlds, static_cast<double*>(d[0]), static_cast<double*>(d[1]), static_cast<double*>(d[2]), nobs,
                      *opt, d_out);
    if (rc) return rc;
    void* host[13] = {nullptr, nullptr, nullptr, out->outcome, out->replans, out->infeasible, out->final_state, out->min_clearance,
                      out->log_state, out->log_q_des, out->log_k, out->log_int, out->log_clearance};
    for (int i = 3; i < 13; i++)
        if (sz[i]) CU(cudaMemcpyAsync(host[i], d[i], sz[i], cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}


int check_clearance(armour_ctx* ctx, int nconf, int nobs) {
    if (!ctx) return ARMOUR_ERR_ARG;
    if (nconf < 1) return fail(ctx, ARMOUR_ERR_ARG, "nconf < 1");
    if (nobs < 0) return fail(ctx, ARMOUR_ERR_ARG, "negative obstacle count");
    if (nobs > ctx->cfg.max_obstacles) return fail(ctx, ARMOUR_ERR_OBSTACLES, "number of obstacles larger than max_obstacles");
    return ARMOUR_OK;
}

}  // namespace

extern "C" {

int armour_batch_rollout_device(armour_ctx* ctx, int nworlds, const double* d_start, const double* d_goal, const double* d_obstacles,
                                int nobs, const armour_rollout_options* opt, const armour_rollout_out* d_out) {
    return rollout_device(ctx, nworlds, d_start, d_goal, d_obstacles, nobs, opt, d_out, false);
}

int armour_batch_rollout(armour_ctx* ctx, int nworlds, const double* start, const double* goal, const double* obstacles, int nobs,
                         const armour_rollout_options* opt, const armour_rollout_out* out) {
    return rollout_host(ctx, nworlds, start, goal, obstacles, nobs, opt, out, false);
}

int armour_armtd_batch_rollout_device(armour_ctx* ctx, int nworlds, const double* d_start, const double* d_goal,
                                      const double* d_obstacles, int nobs, const armour_rollout_options* opt,
                                      const armour_rollout_out* d_out) {
    return rollout_device(ctx, nworlds, d_start, d_goal, d_obstacles, nobs, opt, d_out, true);
}

int armour_armtd_batch_rollout(armour_ctx* ctx, int nworlds, const double* start, const double* goal, const double* obstacles,
                               int nobs, const armour_rollout_options* opt, const armour_rollout_out* out) {
    return rollout_host(ctx, nworlds, start, goal, obstacles, nobs, opt, out, true);
}
int armour_batch_clearance_device(armour_ctx* ctx, int nconf, const double* d_q, const int* d_world, const double* d_obstacles,
                                  int nobs, double* d_clearance, int* d_which) {
    int rc = check_clearance(ctx, nconf, nobs);
    if (rc) return rc;
    if (!d_q || !d_clearance || (nobs > 0 && !d_obstacles)) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    k_clearance<<<nconf, CLEAR_THREADS, 0, ctx->stream>>>(d_q, 1, d_world, d_obstacles, nobs, d_clearance, d_which);
    CU(cudaGetLastError());
    ctx->launches += 1;
    return ARMOUR_OK;
}

int armour_batch_clearance(armour_ctx* ctx, int nconf, const double* q, const int* world, const double* obstacles, int nobs,
                           double* clearance, int* which) {
    int rc = check_clearance(ctx, nconf, nobs);
    if (rc) return rc;
    if (!q || !clearance || (nobs > 0 && !obstacles)) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    int nsets = 1;
    if (world)
        for (int i = 0; i < nconf; i++) {
            if (world[i] < 0) return fail(ctx, ARMOUR_ERR_ARG, "negative obstacle-set index");
            nsets = std::max(nsets, world[i] + 1);
        }
    CU(cudaSetDevice(ctx->cfg.device));
    const size_t nq = size_t(nconf) * NF * 8, nw = world ? size_t(nconf) * 4 : 0, nb = size_t(nsets) * nobs * 12 * 8,
                 nc = size_t(nconf) * 8, nh = which ? size_t(nconf) * 4 : 0;
    void* d[5];  // q, world, obstacles, clearance, which
    rc = stage(ctx, {nq, nw, nb, nc, nh}, d);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(d[0], q, nq, cudaMemcpyHostToDevice, st));
    if (world) CU(cudaMemcpyAsync(d[1], world, nw, cudaMemcpyHostToDevice, st));
    if (nobs > 0) CU(cudaMemcpyAsync(d[2], obstacles, nb, cudaMemcpyHostToDevice, st));
    rc = armour_batch_clearance_device(ctx, nconf, static_cast<double*>(d[0]), static_cast<int*>(d[1]), static_cast<double*>(d[2]), nobs,
                                       static_cast<double*>(d[3]), static_cast<int*>(d[4]));
    if (rc) return rc;
    CU(cudaMemcpyAsync(clearance, d[3], nc, cudaMemcpyDeviceToHost, st));
    if (which) CU(cudaMemcpyAsync(which, d[4], nh, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}

// ---- getters ---------------------------------------------------------------------------------------
int armour_batch_get_torque_radius(armour_ctx* ctx, int nprob, double* out) {
    if (!ctx || !out || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    int rc = fetch_torque_radius(ctx);
    if (rc) return rc;
    std::memcpy(out, ctx->h_torque_radius.data(), size_t(nprob) * NF * ctx->B.T * sizeof(double));
    return ARMOUR_OK;
}
int armour_get_torque_radius(armour_ctx* ctx, double* out) { return armour_batch_get_torque_radius(ctx, 1, out); }

int armour_batch_get_link_independent_generators(armour_ctx* ctx, int nprob, double* out) {
    if (!ctx || !out || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    CU(cudaMemcpyAsync(out, ctx->B.link_gens, size_t(nprob) * ctx->B.T * ctx->B.NJ * 18 * sizeof(double),
                       cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}
int armour_get_link_independent_generators(armour_ctx* ctx, double* out) {
    return armour_batch_get_link_independent_generators(ctx, 1, out);
}

int armour_get_link_sliced_center(armour_ctx* ctx, double* out) {
    if (!ctx || !out || ctx->built_nprob < 1) return ARMOUR_ERR_ARG;
    CU(cudaMemcpyAsync(out, ctx->B.link_sliced, size_t(ctx->B.T) * ctx->B.NJ * 3 * sizeof(double),
                       cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

int armour_batch_get_bounds(armour_ctx* ctx, int nprob, double* g_l, double* g_u) {  // KPR/NLPclass.cu:116-165
    if (!ctx || !g_l || !g_u || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    int rc = fetch_torque_radius(ctx);
    if (rc) return rc;
    const RobotConstants& R = ctx->rc;
    const int T = ctx->B.T, NJ = ctx->B.NJ, O = ctx->B.O, m = ctx->B.m();
    for (int p = 0; p < nprob; p++) {
        double* gl = g_l + size_t(p) * m;
        double* gu = g_u + size_t(p) * m;
        const double* tr = ctx->h_torque_radius.data() + size_t(p) * NF * T;
        for (int t = 0; t < T; t++)
            for (int j = 0; j < NF; j++) {
                gl[t * NF + j] = -R.torque_limits[j] + tr[j * T + t];
                gu[t * NF + j] = R.torque_limits[j] - tr[j * T + t];
            }
        int off = NF * T;
        for (int i = off; i < off + T * NJ * O; i++) {
            gl[i] = -1e19;
            gu[i] = 0;
        }
        off += T * NJ * O;
        for (int rep = 0; rep < 2; rep++, off += NF)
            for (int i = 0; i < NF; i++) {
                gl[off + i] = R.state_limits_lb[i] + R.qe;
                gu[off + i] = R.state_limits_ub[i] - R.qe;
            }
        for (int rep = 0; rep < 2; rep++, off += NF)
            for (int i = 0; i < NF; i++) {
                gl[off + i] = -R.speed_limits[i] + R.qde;
                gu[off + i] = R.speed_limits[i] - R.qde;
            }
    }
    return ARMOUR_OK;
}
int armour_get_bounds(armour_ctx* ctx, double* g_l, double* g_u) { return armour_batch_get_bounds(ctx, 1, g_l, g_u); }

int armour_verdict(armour_ctx* ctx, const double* g, int* feasible, int* first_violation) {  // KPR/NLPclass.cu:449-537
    if (!ctx || !g || !feasible || ctx->built_nprob < 1) return ARMOUR_ERR_ARG;
    int rc = fetch_torque_radius(ctx);
    if (rc) return rc;
    const RobotConstants& R = ctx->rc;
    const int T = ctx->B.T, NJ = ctx->B.NJ, O = ctx->B.O;
    const double* tr = ctx->h_torque_radius.data();
    auto done = [&](int ok, int row) {
        *feasible = ok;
        if (first_violation) *first_violation = row;
        return ARMOUR_OK;
    };
    for (int t = 0; t < T; t++)
        for (int j = 0; j < NF; j++) {
            const double v = g[t * NF + j];
            if (v < -R.torque_limits[j] + tr[j * T + t] - R.torque_violation_threshold ||
                v > R.torque_limits[j] - tr[j * T + t] + R.torque_violation_threshold)
                return done(0, t * NF + j);
        }
    int off = NF * T;
    for (int i = 0; i < NJ * T * O; i++)
        if (g[off + i] > R.collision_violation_threshold) return done(0, off + i);
    off += NJ * T * O;
    for (int rep = 0; rep < 2; rep++, off += NF)
        for (int i = 0; i < NF; i++)
            if (g[off + i] < R.state_limits_lb[i] + R.qe || g[off + i] > R.state_limits_ub[i] - R.qe)
                return done(0, off + i);
    for (int rep = 0; rep < 2; rep++, off += NF)
        for (int i = 0; i < NF; i++)
            if (g[off + i] < -R.speed_limits[i] + R.qde || g[off + i] > R.speed_limits[i] - R.qde)
                return done(0, off + i);
    return done(1, -1);
}

int armour_cost(armour_ctx* ctx, const double* q_des, const double* k, double* obj, double* grad) {
    if (!ctx || !q_des || !k || ctx->built_nprob < 1 || ctx->h_q0.empty()) return ARMOUR_ERR_ARG;
    const RobotConstants& R = ctx->rc;
    auto wrap = [](double a) {  // KPR/NLPclass.cu:6-15
        while (a < -M_PI) a += 2 * M_PI;
        while (a > M_PI) a -= 2 * M_PI;
        return a;
    };
    const double tp = R.t_plan, D = R.duration;
    double qp[NF];
    for (int i = 0; i < NF; i++)
        qp[i] = bez_q(ctx->h_q0[i], ctx->h_qd0[i] * D, ctx->h_qdd0[i] * D * D, R.k_range[i] * k[i], tp);
    if (obj) {  // KPR/NLPclass.cu:222-233
        double v = pw2(wrap(q_des[0] - qp[0])) + pw2(wrap(q_des[2] - qp[2])) + pw2(wrap(q_des[4] - qp[4])) +
                   pw2(wrap(q_des[6] - qp[6])) + pw2(q_des[1] - qp[1]) + pw2(q_des[3] - qp[3]) + pw2(q_des[5] - qp[5]);
        *obj = v * R.cost_scale;
    }
    if (grad) {  // KPR/NLPclass.cu:252-264
        for (int i = 0; i < NF; i++) {
            const double dk = pw3(tp) * (6 * pw2(tp) - 15 * tp + 10) * R.k_range[i];
            grad[i] = (i % 2 == 0) ? (2 * wrap(qp[i] - q_des[i]) * dk) : (2 * (qp[i] - q_des[i]) * dk);
            grad[i] *= R.cost_scale;
        }
    }
    return ARMOUR_OK;
}

// ---- reach-set tables ------------------------------------------------------------------------------
int armour_export_reachsets(armour_ctx* ctx, int prob, armour_reachset_tables* out) {
    if (!ctx || !out || prob < 0 || prob >= ctx->built_nprob) return ARMOUR_ERR_ARG;
    const Batch& B = ctx->B;
    const size_t T = B.T, NJ = B.NJ;
    if (out->cap_link < B.capL || out->cap_u < B.capU) return fail(ctx, ARMOUR_ERR_ARG, "export caps too small");
    std::vector<uint16_t> lk(T * NJ * B.capL), uk(T * NF * B.capU);
    std::vector<double> lg(T * NJ * B.capL * 3), ug(T * NF * B.capU);
    cudaStream_t st = ctx->stream;
#define D2H(dst, src, n) CU(cudaMemcpyAsync(dst, src, (n), cudaMemcpyDeviceToHost, st))
    D2H(out->link_n, B.link_n + prob * T * NJ, T * NJ * sizeof(int));
    D2H(out->link_center, B.link_c + prob * T * NJ * 3, T * NJ * 3 * sizeof(double));
    D2H(lk.data(), B.link_key + prob * T * NJ * B.capL, lk.size() * sizeof(uint16_t));
    D2H(lg.data(), B.link_g + prob * T * NJ * B.capL * 3, lg.size() * sizeof(double));
    D2H(out->u_n, B.u_n + prob * T * NF, T * NF * sizeof(int));
    D2H(out->u_center, B.u_c + prob * T * NF, T * NF * sizeof(double));
    D2H(uk.data(), B.u_key + prob * T * NF * B.capU, uk.size() * sizeof(uint16_t));
    D2H(ug.data(), B.u_g + prob * T * NF * B.capU, ug.size() * sizeof(double));
    if (out->u_radius) D2H(out->u_radius, B.u_r + prob * T * NF, T * NF * sizeof(double));
    if (out->torque_radius) D2H(out->torque_radius, B.torque_radius + prob * NF * T, NF * T * sizeof(double));
    if (out->link_gens) D2H(out->link_gens, B.link_gens + prob * T * NJ * 18, T * NJ * 18 * sizeof(double));
#undef D2H
    CU(cudaStreamSynchronize(st));
    // entries past the monomial count are padding: export them as zero
    for (size_t i = 0; i < T * NJ; i++)
        for (int mI = 0; mI < out->cap_link; mI++) {
            const bool valid = mI < out->link_n[i] && mI < B.capL;
            out->link_key[i * out->cap_link + mI] = valid ? lk[i * B.capL + mI] : 0;
            for (int e = 0; e < 3; e++)
                out->link_coeff[(i * out->cap_link + mI) * 3 + e] = valid ? lg[(i * B.capL + mI) * 3 + e] : 0.0;
        }
    for (size_t i = 0; i < T * NF; i++)
        for (int mI = 0; mI < out->cap_u; mI++) {
            const bool valid = mI < out->u_n[i] && mI < B.capU;
            out->u_key[i * out->cap_u + mI] = valid ? uk[i * B.capU + mI] : 0;
            out->u_coeff[i * out->cap_u + mI] = valid ? ug[i * B.capU + mI] : 0.0;
        }
    return ARMOUR_OK;
}

int armour_import_reachsets(armour_ctx* ctx, int prob, int nprob_total, const armour_reachset_tables* in,
                            const double* q0, const double* qd0, const double* qdd0, const double* obstacles, int nobs) {
    int rc = check_batch(ctx, nprob_total, nobs);
    if (rc) return rc;
    if (!in || !in->u_radius || !in->torque_radius || !in->link_gens || !q0 || !qd0 || !qdd0 || prob < 0 ||
        prob >= nprob_total)
        return ARMOUR_ERR_ARG;
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    if (prob == 0 || ctx->B.O != nobs || ctx->B.nprob != nprob_total) {
        rc = ensure_obstacle_buffers(ctx, nprob_total, nobs);
        if (rc) return rc;
        ctx->B.O = nobs;
        ctx->B.nprob = nprob_total;
    }
    if (prob == 0) ctx->B.epoch++;  // imported tables: no build failure can be pending
    const Batch& B = ctx->B;
    const size_t T = B.T, NJ = B.NJ, P = size_t(ctx->cfg.max_problems);
    std::vector<uint16_t> lk(T * NJ * B.capL, 0), uk(T * NF * B.capU, 0);
    std::vector<double> lg(T * NJ * B.capL * 3, 0.0), ug(T * NF * B.capU, 0.0);
    for (size_t i = 0; i < T * NJ; i++) {
        if (in->link_n[i] > B.capL) return fail(ctx, ARMOUR_ERR_CAPACITY, "imported link table exceeds cap_link_monomials");
        for (int mI = 0; mI < in->link_n[i]; mI++) {
            lk[i * B.capL + mI] = uint16_t(in->link_key[i * in->cap_link + mI]);
            for (int e = 0; e < 3; e++) lg[(i * B.capL + mI) * 3 + e] = in->link_coeff[(i * in->cap_link + mI) * 3 + e];
        }
    }
    for (size_t i = 0; i < T * NF; i++) {
        if (in->u_n[i] > B.capU) return fail(ctx, ARMOUR_ERR_CAPACITY, "imported torque table exceeds cap_torque_monomials");
        for (int mI = 0; mI < in->u_n[i]; mI++) {
            uk[i * B.capU + mI] = uint16_t(in->u_key[i * in->cap_u + mI]);
            ug[i * B.capU + mI] = in->u_coeff[i * in->cap_u + mI];
        }
    }
    cudaStream_t st = ctx->stream;
#define H2D(dst, src, n) CU(cudaMemcpyAsync(dst, src, (n), cudaMemcpyHostToDevice, st))
    H2D(B.link_n + prob * T * NJ, in->link_n, T * NJ * sizeof(int));
    H2D(B.link_c + prob * T * NJ * 3, in->link_center, T * NJ * 3 * sizeof(double));
    H2D(B.link_key + prob * T * NJ * B.capL, lk.data(), lk.size() * sizeof(uint16_t));
    H2D(B.link_g + prob * T * NJ * B.capL * 3, lg.data(), lg.size() * sizeof(double));
    H2D(B.u_n + prob * T * NF, in->u_n, T * NF * sizeof(int));
    H2D(B.u_c + prob * T * NF, in->u_center, T * NF * sizeof(double));
    H2D(B.u_key + prob * T * NF * B.capU, uk.data(), uk.size() * sizeof(uint16_t));
    H2D(B.u_g + prob * T * NF * B.capU, ug.data(), ug.size() * sizeof(double));
    H2D(B.torque_radius + prob * NF * T, in->torque_radius, NF * T * sizeof(double));
    H2D(B.link_gens + prob * T * NJ * 18, in->link_gens, T * NJ * 18 * sizeof(double));
    std::vector<double> lr(T * NJ * 3);
    for (size_t i = 0; i < T * NJ; i++)
        for (int e = 0; e < 3; e++) lr[i * 3 + e] = in->link_gens[i * 18 + e + (3 + e) * 3];
    H2D(B.link_r + prob * T * NJ * 3, lr.data(), lr.size() * sizeof(double));
    H2D(B.u_r + prob * T * NF, in->u_radius, T * NF * sizeof(double));
    H2D(ctx->d_in.get() + prob * NF, q0, NF * sizeof(double));
    H2D(ctx->d_in.get() + P * NF + prob * NF, qd0, NF * sizeof(double));
    H2D(ctx->d_in.get() + 2 * P * NF + prob * NF, qdd0, NF * sizeof(double));
    if (nobs > 0) H2D(ctx->d_obs.get() + size_t(prob) * nobs * 12, obstacles, size_t(nobs) * 12 * sizeof(double));
#undef H2D
    CU(cudaStreamSynchronize(st));  // the staging vectors die at return
    if (prob == nprob_total - 1) {
        if (nobs > 0) CU(cudaMemsetAsync(ctx->B.hp_slow, 0, size_t(nprob_total) * sizeof(int), ctx->stream));
        CU(launch_hyperplanes(ctx->B, ctx->stream));
        ctx->launches += (nobs > 0);
        CU(launch_pack_image(ctx->B, ctx->stream));
        ctx->launches++;
        ctx->built_nprob = nprob_total;
        ctx->h_torque_valid = false;
    }
    if (prob == 0) {
        ctx->h_q0.assign(q0, q0 + NF);
        ctx->h_qd0.assign(qd0, qd0 + NF);
        ctx->h_qdd0.assign(qdd0, qdd0 + NF);
    }
    return ARMOUR_OK;
}


// ---- ARMTD comparison planner (SURVEY.md 8f-3; csrc/armtd.cuh) ---------------------------------------------------------------
// A batch of nprob problems (worlds) per context; the single-problem calls are batches of one.
}  // extern "C"

namespace {

int armtd_ctx_create(const armour_config* cfg_in, bool batch, armour_ctx** out) {
    if (!out) return ARMOUR_ERR_ARG;
    armour_config cfg;
    if (cfg_in) {
        cfg = *cfg_in;
    } else {
        int rc = armour_config_default(&cfg);
        if (rc) return rc;
    }
    cfg.num_time_steps = ARMTD_T_PADDED;  // 100 intervals of KPA + 4 padding intervals (chunks of 8)
    if (!batch) cfg.max_problems = 1;
    cfg.robot_model = 0;  // KPA/Parameters.h:6: KinovaWithoutGripperInfo.h
    armour_ctx* ctx = nullptr;
    int rc = armour_ctx_create(&cfg, &ctx);
    if (rc) return rc;
    const size_t P = size_t(ctx->cfg.max_problems);
    if (ctx->d_jrs.reserve(P * ARMTD_T_PADDED * NF * 6) != cudaSuccess ||
        ctx->d_armtd_in.reserve(P * NF * 4 + P * 6 * NF * ARMTD_T) != cudaSuccess ||
        cudaMemsetAsync(ctx->d_armtd_in.get(), 0, P * NF * 2 * sizeof(double), ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess) {
        armour_ctx_destroy(ctx);
        return ARMOUR_ERR_NOMEM;
    }
    ctx->d_krange = ctx->d_armtd_in.get();
    ctx->d_zero = ctx->d_krange + P * NF;
    ctx->d_cs = ctx->d_zero + P * NF;
    ctx->d_jrs_raw = ctx->d_cs + P * NF * 2;
    ctx->armtd = true;
    ctx->B.jrs_ext = ctx->d_jrs.get();
    *out = ctx;
    return ARMOUR_OK;
}

int check_armtd_batch(armour_ctx* ctx, int nprob, int nobs) {
    if (!ctx) return ARMOUR_ERR_ARG;
    if (!ctx->armtd) return fail(ctx, ARMOUR_ERR_STATE, "not an ARMTD context (armour_armtd_ctx_create / armour_armtd_batch_ctx_create)");
    return check_batch(ctx, nprob, nobs);
}

// problems [0, nprob) of the last build were evaluated / solved before?  (ARMOUR_ERR_STATE as in the main planner's calls)
int check_armtd_built(armour_ctx* ctx, int nprob, const char* what) {
    if (!ctx->armtd) return fail(ctx, ARMOUR_ERR_STATE, "not an ARMTD context (armour_armtd_ctx_create / armour_armtd_batch_ctx_create)");
    if (nprob < 1 || nprob > ctx->built_nprob) return fail(ctx, ARMOUR_ERR_STATE, std::string(what) + " before armour_armtd_build");
    return ARMOUR_OK;
}

int ensure_armtd_buffers(armour_ctx* ctx, int nprob, bool need_jac) {
    const size_t ma = size_t(nprob) * armtd_m(ctx->B.NJ, ctx->B.O);
    CU(ctx->d_ga.reserve(ma));
    if (need_jac) CU(ctx->d_ja.reserve(ma * NF));
    return ARMOUR_OK;
}

// one evaluation of the problems of Bb at d_k in KPA's layout: k_constraints into the context's full-layout buffers (sized by
// the caller), then k_armtd_assemble (d_g / d_jac may be nullptr; with d_jac == nullptr no Jacobian is computed).  Launches
// 2 + (O > 0) kernels.
int armtd_eval_launch(armour_ctx* ctx, const Batch& Bb, const double* d_k, double* d_g, double* d_jac) {
    CU(launch_constraints(Bb, d_k, ctx->d_g.get(), d_jac ? ctx->d_jac.get() : nullptr, ctx->stream));
    CU(launch_armtd_assemble(Bb, ctx->d_krange, d_k, ctx->d_g.get(), ctx->d_jac.get(), d_g, d_jac, ctx->stream));
    return ARMOUR_OK;
}

// host copies of q0, qd0 and k_range of the built problems (the cost is host arithmetic)
int fetch_armtd_inputs(armour_ctx* ctx) {
    const size_t n = size_t(ctx->built_nprob) * NF, P = size_t(ctx->cfg.max_problems);
    if (ctx->h_q0.size() >= n && ctx->h_qd0.size() >= n && ctx->h_krange.size() >= n) return ARMOUR_OK;
    ctx->h_q0.resize(n);
    ctx->h_qd0.resize(n);
    ctx->h_qdd0.assign(n, 0.0);
    ctx->h_krange.resize(n);
    CU(cudaMemcpyAsync(ctx->h_q0.data(), ctx->d_in.get(), n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(ctx->h_qd0.data(), ctx->d_in.get() + P * NF, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpyAsync(ctx->h_krange.data(), ctx->d_krange, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}

}  // namespace

extern "C" {

int armour_armtd_ctx_create(const armour_config* cfg, armour_ctx** out) { return armtd_ctx_create(cfg, false, out); }
int armour_armtd_batch_ctx_create(const armour_config* cfg, armour_ctx** out) { return armtd_ctx_create(cfg, true, out); }

int armour_armtd_num_constraints(const armour_ctx* ctx) {
    if (!ctx || !ctx->armtd) return ARMOUR_ERR_ARG;
    return armtd_m(ctx->B.NJ, ctx->B.O);
}

int armour_armtd_batch_build_device(armour_ctx* ctx, int nprob, const double* d_q0, const double* d_qd0, const double* d_jrs,
                                    const double* d_k_range, const double* d_obstacles, int nobs, const double* d_sincos) {
    int rc = check_armtd_batch(ctx, nprob, nobs);
    if (rc) return rc;
    if (!d_q0 || !d_qd0 || !d_jrs || !d_k_range || (nobs > 0 && !d_obstacles)) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    const int n = nprob * ARMTD_T_PADDED * NF;
    k_armtd_jrs<<<(n + 255) / 256, 256, 0, ctx->stream>>>(nprob, d_q0, d_sincos, d_jrs, ctx->d_jrs.get());
    CU(cudaGetLastError());
    ctx->launches++;
    CU(cudaMemcpyAsync(ctx->d_krange, d_k_range, size_t(nprob) * NF * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    ctx->h_krange.clear();
    return armour_batch_reachsets_build_device(ctx, nprob, d_q0, d_qd0, ctx->d_zero, d_obstacles, nobs);
}

int armour_armtd_offline_jrs_device(armour_ctx* ctx, int n, const double* d_qd0, const double* d_k_range, double* d_jrs) {
    if (!ctx) return ARMOUR_ERR_ARG;
    if (!ctx->armtd) return fail(ctx, ARMOUR_ERR_STATE, "not an ARMTD context (armour_armtd_ctx_create / armour_armtd_batch_ctx_create)");
    if (n < 1) return fail(ctx, ARMOUR_ERR_ARG, "n < 1");
    if (!d_qd0 || !d_k_range || !d_jrs) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    CU(launch_armtd_offline_jrs(n, d_qd0, d_k_range, nullptr, d_jrs, ctx->stream));
    ctx->launches++;
    return ARMOUR_OK;
}

int armour_armtd_offline_jrs(armour_ctx* ctx, int n, const double* qd0, const double* k_range, double* jrs) {
    if (!ctx) return ARMOUR_ERR_ARG;
    if (!ctx->armtd) return fail(ctx, ARMOUR_ERR_STATE, "not an ARMTD context (armour_armtd_ctx_create / armour_armtd_batch_ctx_create)");
    if (n < 1) return fail(ctx, ARMOUR_ERR_ARG, "n < 1");
    if (!qd0 || !k_range || !jrs) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    CU(cudaSetDevice(ctx->cfg.device));
    const size_t nk = size_t(n) * NF * sizeof(double), nj = size_t(n) * 6 * NF * ARMTD_T * sizeof(double);
    void* d[3];  // qd0, k_range, jrs
    int rc = stage(ctx, {nk, nk, nj}, d);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(d[0], qd0, nk, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d[1], k_range, nk, cudaMemcpyHostToDevice, st));
    rc = armour_armtd_offline_jrs_device(ctx, n, static_cast<double*>(d[0]), static_cast<double*>(d[1]), static_cast<double*>(d[2]));
    if (rc) return rc;
    CU(cudaMemcpyAsync(jrs, d[2], nj, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}

int armour_armtd_batch_build(armour_ctx* ctx, int nprob, const double* q0, const double* qd0, const double* jrs,
                             const double* k_range, const double* obstacles, int nobs) {
    int rc = check_armtd_batch(ctx, nprob, nobs);
    if (rc) return rc;
    if (!q0 || !qd0 || !jrs || !k_range || (nobs > 0 && !obstacles)) return fail(ctx, ARMOUR_ERR_ARG, "null input");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    // cos q0 / sin q0 with the host's libm, as the reference's ConstantAccelerationCurve constructor (KPA/Trajectory.cu:29-62)
    const size_t n = size_t(nprob) * NF;
    std::vector<double> cs(2 * n);
    for (size_t x = 0; x < n; x++) {
        cs[2 * x] = std::cos(q0[x]);
        cs[2 * x + 1] = std::sin(q0[x]);
    }
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(ctx->d_cs, cs.data(), cs.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_jrs_raw, jrs, n * 6 * ARMTD_T * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ctx->d_krange, k_range, n * sizeof(double), cudaMemcpyHostToDevice, st));
    const int nt = nprob * ARMTD_T_PADDED * NF;
    k_armtd_jrs<<<(nt + 255) / 256, 256, 0, st>>>(nprob, nullptr, ctx->d_cs, ctx->d_jrs_raw, ctx->d_jrs.get());
    CU(cudaGetLastError());
    ctx->launches++;
    ctx->h_krange.assign(k_range, k_range + n);
    const std::vector<double> zero(n, 0.0);
    rc = armour_batch_reachsets_build(ctx, nprob, q0, qd0, zero.data(), obstacles, nobs);
    if (rc != ARMOUR_OK && rc != ARMOUR_ERR_CAPACITY) cudaStreamSynchronize(st);  // (the staging vectors die at return)
    return rc;
}

int armour_armtd_build(armour_ctx* ctx, const double* q0, const double* qd0, const double* jrs, const double* k_range,
                       const double* obstacles, int nobs) {
    if (!ctx || !q0 || !qd0 || !jrs || !k_range) return ARMOUR_ERR_ARG;
    return armour_armtd_batch_build(ctx, 1, q0, qd0, jrs, k_range, obstacles, nobs);
}

int armour_armtd_batch_eval_device(armour_ctx* ctx, int nprob, const double* d_k, double* d_g, double* d_values) {
    if (!ctx || !d_k || (!d_g && !d_values)) return ARMOUR_ERR_ARG;
    int rc = check_armtd_built(ctx, nprob, "evaluate");
    if (rc) return rc;
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    rc = ensure_eval_buffers(ctx, size_t(nprob) * ctx->B.m(), true, d_values != nullptr);
    if (rc) return rc;
    Batch B = ctx->B;
    B.nprob = nprob;
    rc = armtd_eval_launch(ctx, B, d_k, d_g, d_values);
    ctx->launches += 2 + (B.O > 0);
    return rc;
}

int armour_armtd_batch_eval(armour_ctx* ctx, int nprob, const double* k, double* g, double* values) {
    if (!ctx || !k || (!g && !values)) return ARMOUR_ERR_ARG;
    int rc = check_armtd_built(ctx, nprob, "evaluate");
    if (rc) return rc;
    CU(cudaSetDevice(ctx->cfg.device));
    rc = ensure_armtd_buffers(ctx, nprob, values != nullptr);
    if (rc) return rc;
    const size_t ma = size_t(nprob) * armtd_m(ctx->B.NJ, ctx->B.O);
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(ctx->d_k.get(), k, size_t(nprob) * NF * sizeof(double), cudaMemcpyHostToDevice, st));
    rc = armour_armtd_batch_eval_device(ctx, nprob, ctx->d_k.get(), g ? ctx->d_ga.get() : nullptr, values ? ctx->d_ja.get() : nullptr);
    if (rc) return rc;
    if (g) CU(cudaMemcpyAsync(g, ctx->d_ga.get(), ma * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (values) CU(cudaMemcpyAsync(values, ctx->d_ja.get(), ma * NF * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ARMOUR_OK;
}

int armour_armtd_eval(armour_ctx* ctx, const double* k, double* g, double* values) {
    return armour_armtd_batch_eval(ctx, 1, k, g, values);
}

int armour_armtd_get_bounds(armour_ctx* ctx, double* g_l, double* g_u) {  // KPA/NLPclass.cu:75-142
    if (!ctx || !g_l || !g_u || !ctx->armtd || ctx->built_nprob < 1) return ARMOUR_ERR_ARG;
    const RobotConstants& R = ctx->rc;
    int off = ctx->B.NJ * ARMTD_T * ctx->B.O;
    for (int i = 0; i < off; i++) {
        g_l[i] = -1e19;
        g_u[i] = 0;
    }
    for (int rep = 0; rep < 2; rep++, off += NF)
        for (int i = 0; i < NF; i++) {
            g_l[off + i] = R.state_limits_lb[i] + R.qe;
            g_u[off + i] = R.state_limits_ub[i] - R.qe;
        }
    for (int rep = 0; rep < 2; rep++, off += NF)
        for (int i = 0; i < NF; i++) {
            g_l[off + i] = -R.speed_limits[i] + R.qde;
            g_u[off + i] = R.speed_limits[i] - R.qde;
        }
    return ARMOUR_OK;
}

int armour_armtd_batch_verdict_device(armour_ctx* ctx, int nprob, const double* d_g, int* d_feasible, int* d_first) {
    if (!ctx || !d_g || !d_feasible || !d_first) return ARMOUR_ERR_ARG;
    int rc = check_armtd_built(ctx, nprob, "verdict");
    if (rc) return rc;
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    k_armtd_verdict<<<nprob, 256, 0, ctx->stream>>>(ctx->B.NJ, ctx->B.O, d_g, d_feasible, d_first);
    CU(cudaGetLastError());
    ctx->launches++;
    return ARMOUR_OK;
}

int armour_armtd_verdict(armour_ctx* ctx, const double* g, int* feasible, int* first_violation) {  // KPA/NLPclass.cu:366-455
    if (!ctx || !g || !feasible || !ctx->armtd || ctx->built_nprob < 1) return ARMOUR_ERR_ARG;
    CU(cudaSetDevice(ctx->cfg.device));
    int rc = ensure_armtd_buffers(ctx, 1, false);
    if (rc) return rc;
    cudaStream_t st = ctx->stream;
    CU(cudaMemcpyAsync(ctx->d_ga.get(), g, size_t(armtd_m(ctx->B.NJ, ctx->B.O)) * sizeof(double), cudaMemcpyHostToDevice, st));
    rc = armour_armtd_batch_verdict_device(ctx, 1, ctx->d_ga.get(), ctx->d_verdict.get(), ctx->d_verdict.get() + 1);
    if (rc) return rc;
    int v[2];
    CU(cudaMemcpyAsync(v, ctx->d_verdict.get(), sizeof(v), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *feasible = v[0];
    if (first_violation) *first_violation = v[1];
    return ARMOUR_OK;
}

int armour_armtd_batch_cost(armour_ctx* ctx, int nprob, const double* q_des, const double* k, double* obj, double* grad) {
    if (!ctx || !q_des || !k || !ctx->armtd || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    int rc = fetch_armtd_inputs(ctx);
    if (rc) return rc;
    for (int p = 0; p < nprob; p++) {
        const size_t o = size_t(p) * NF;
        const double f = armtd_cost(ctx->h_q0.data() + o, ctx->h_qd0.data() + o, ctx->h_krange.data() + o, q_des + o, k + o,
                                    ctx->rc.cost_scale, grad ? grad + o : nullptr);
        if (obj) obj[p] = f;
    }
    return ARMOUR_OK;
}

int armour_armtd_cost(armour_ctx* ctx, const double* q_des, const double* k, double* obj, double* grad) {  // KPA/NLPclass.cu:178-243
    return armour_armtd_batch_cost(ctx, 1, q_des, k, obj, grad);
}

int armour_armtd_batch_solve_device(armour_ctx* ctx, int nprob, const double* d_q_des, const armour_solver_options* opt_in,
                                    double* d_k_opt, int* d_feasible, int* d_first, int* d_iters) {
    if (!ctx || !d_q_des || !d_k_opt || !d_feasible || !d_first) return ARMOUR_ERR_ARG;
    int rc = check_armtd_built(ctx, nprob, "solve");
    if (rc) return rc;
    armour_solver_options opt;
    armour_solver_options_default(&opt);
    opt.tol = 1e-7;  // IPOPT_OPTIMIZATION_TOLERANCE of KPA (KPA/Parameters.h:43), as armtd_main sets it
    if (opt_in) opt = *opt_in;
    if (opt.max_iter < 1 || !(opt.tol > 0) || opt.qp_sweeps < 1) return fail(ctx, ARMOUR_ERR_ARG, "solver options");
    { int rc_e = enter(ctx); if (rc_e) return rc_e; }
    rc = ensure_eval_buffers(ctx, size_t(nprob) * ctx->B.m(), true, true);
    if (rc) return rc;
    rc = ensure_armtd_buffers(ctx, nprob, true);
    if (rc) return rc;
    auto eval = [ctx](const Batch& Bb, const double* x, double* g, double* jac) { return armtd_eval_launch(ctx, Bb, x, g, jac); };
    auto verdict = [ctx, nprob](const double* g, int* feasible, int* first) {
        k_armtd_verdict<<<nprob, 256, 0, ctx->stream>>>(ctx->B.NJ, ctx->B.O, g, feasible, first);
        CU(cudaGetLastError());
        return int(ARMOUR_OK);
    };
    return run_solver(ctx, nprob, d_q_des, opt, ArmtdNlp{ctx->d_krange}, armtd_m(ctx->B.NJ, ctx->B.O), ctx->d_ga.get(),
                      ctx->d_ja.get(), eval, 2 + (ctx->B.O > 0), verdict, d_k_opt, d_feasible, d_first, d_iters);
}

int armour_armtd_batch_solve(armour_ctx* ctx, int nprob, const double* q_des, const armour_solver_options* opt, double* k_opt,
                             int* feasible, int* first_violation, int* iterations) {
    if (!ctx || !q_des || !k_opt || !feasible) return ARMOUR_ERR_ARG;
    int rc = check_armtd_built(ctx, nprob, "solve");
    if (rc) return rc;
    return solve_from_host(ctx, nprob, q_des, opt, k_opt, feasible, first_violation, iterations, armour_armtd_batch_solve_device);
}

// armour_joint_position_center.out / armour_joint_position_radius.out of KPA/armtd_main.cu:232-256: [100][NJ][3] and [100][NJ][18]
int armour_armtd_get_link_sliced_center(armour_ctx* ctx, double* out) {
    if (!ctx || !out || !ctx->armtd || ctx->built_nprob < 1) return ARMOUR_ERR_ARG;
    CU(cudaMemcpyAsync(out, ctx->B.link_sliced, size_t(ARMTD_T) * ctx->B.NJ * 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}
int armour_armtd_batch_get_link_independent_generators(armour_ctx* ctx, int nprob, double* out) {
    if (!ctx || !out || !ctx->armtd || nprob < 1 || nprob > ctx->built_nprob) return ARMOUR_ERR_ARG;
    const size_t row = size_t(ctx->B.NJ) * 18 * sizeof(double);  // one interval
    // the 100 intervals of every problem, without the padding intervals
    CU(cudaMemcpy2DAsync(out, ARMTD_T * row, ctx->B.link_gens, ARMTD_T_PADDED * row, ARMTD_T * row, size_t(nprob),
                         cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return ARMOUR_OK;
}
int armour_armtd_get_link_independent_generators(armour_ctx* ctx, double* out) {
    return armour_armtd_batch_get_link_independent_generators(ctx, 1, out);
}

}  // extern "C"
