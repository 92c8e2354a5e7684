// blsgpu.cu — host side of the C ABI declared in include/blsgpu.h: context, staging, launch sequence.
// Everything that computes runs in the kernels of kernels.cuh / msm.cuh; this file only moves bytes and
// launches.  There is no CPU implementation of any operation behind these entry points.
#include <cuda_runtime.h>
#include <limits.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <functional>
#include <string>
#include <map>
#include <vector>
#include "../../include/blsgpu.h"
#include "kernels.cuh"
#include "msm.cuh"
#include "fpprog.hpp"
#include "route.hpp"

using namespace bls;

enum { ST_SCALARS = 0, ST_G2MUL, ST_G2SUM, ST_HASH, ST_G1MUL, ST_AFFINE, ST_LINES, ST_ACC, ST_GTPROD, ST_PARTIAL, ST_FINAL, ST_COUNT };
static const char *STAGE_NAMES[ST_COUNT] = {"rlc_scalars", "g2_mul64", "g2_sum", "hash_to_g2", "g1_mul64", "pairs_affine",
                                            "miller_lines", "miller_acc", "gt_product", "partial", "final_exp"};
static_assert(route::ACC_BLOCK == BLS_ACC_BS && ST_ACC == ST_LINES + 1 && ST_GTPROD == ST_LINES + 2 && ST_PARTIAL == ST_LINES + 3,
              "route.hpp / miller_ws layout");
static_assert(route::LB_BLOCKS == BLS_LB_BLOCKS, "route.hpp plan_msm sizes the chunk grid for the BLS_LB occupancy");

// device programs (fpprog.hpp) kept in blsgpu_ctx::progs, by kind and a key (see get_prog)
enum prog_kind { PROG_COMBINE, PROG_FINAL, PROG_NORM, PROG_SET, PROG_PRODUCT, PROG_MSM_HORNER_G1, PROG_MSM_HORNER_G2 };

// Buffers, stream and stage events of one multi-Miller loop (run_miller)
struct miller_ws {
    route::miller_caps caps = {}; // sizes of the buffers below
    uint32_t *lines = nullptr;    // 68 x 72 words x caps.lines_cap
    fp12 *F = nullptr;            // per-segment block products, nseg rows
    fp12 *F2 = nullptr;           // second-level block products
    fp12 *seg = nullptr;          // 64 segment products
    fp *small_lines = nullptr;    // 68 x 6 field elements per pair (small-batch route), allocated on first use
    cudaStream_t stream = nullptr;
    cudaEvent_t *ev = nullptr;    // begin/end pairs of miller_lines, miller_acc, gt_product, partial
};

static void miller_ws_free(miller_ws &ws) {
    cudaFree(ws.lines); cudaFree(ws.F); cudaFree(ws.F2); cudaFree(ws.seg); cudaFree(ws.small_lines);
    ws.lines = nullptr; ws.F = ws.F2 = ws.seg = nullptr; ws.small_lines = nullptr;
}

// lines, F, F2 and seg of ws, sized from ws.caps; all or none: on failure ws is left without buffers
static cudaError_t miller_ws_alloc(miller_ws &ws) {
    cudaError_t e = cudaMalloc((void **)&ws.lines, (size_t)ML_NLINES * ML_LINE_WORDS * 4 * ws.caps.lines_cap);
    if (e == cudaSuccess) e = cudaMalloc((void **)&ws.F, ws.caps.f_cap * sizeof(fp12));
    if (e == cudaSuccess) e = cudaMalloc((void **)&ws.F2, ws.caps.f2_cap * sizeof(fp12));
    if (e == cudaSuccess) e = cudaMalloc((void **)&ws.seg, 64 * sizeof(fp12));
    if (e != cudaSuccess) miller_ws_free(ws);
    return e;
}

enum { H2D_SLICES = 4 };

struct blsgpu_ctx {
    int device = 0;
    size_t cap = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // device buffers
    sigset *d_sets = nullptr;
    uint64_t *d_r = nullptr;
    g2_jac *d_H = nullptr;
    g1_jac *d_Pj = nullptr;
    g2_aff *d_Q = nullptr;
    g1_aff *d_P = nullptr;
    g2_jac *d_S = nullptr;
    miller_ws ml;                 // the Miller loop over the batch's pairs: on `stream`, events of ST_LINES..ST_PARTIAL
    // the one-pair Miller loop of (S, -G1) when it runs on the side stream beside the main loop (run_partial_impl):
    // buffers allocated on first use, events in ev_scratch
    miller_ws ml_sig;
    bool acc_team = true;         // six-lane team accumulation (acc_team.cuh) vs one thread per group
    fp12 *d_partials = nullptr;   // 64 slots
    uint8_t *d_gtb = nullptr;     // 576 canonical GT bytes
    int *d_flags = nullptr;       // [0] pk infinity, [1] is_one
    unsigned long long *d_dbg = nullptr;                     // BLSGPU_DEBUG_CHAIN: timestamps of the scalar chain
    void *d_misc = nullptr;       // scratch for aggregate / hash API
    size_t misc_bytes = 0;
    void *d_misc2 = nullptr;      // small result scratch (MSM output)
    uint8_t *h_pinned = nullptr;  // 4 KiB pinned for small D2H results
    cudaEvent_t ev[2 * ST_COUNT + 5];                        // stage begin/end pairs + fork/join/G1-ready
    bool ev_valid[2 * ST_COUNT + 5];
    cudaEvent_t ev_scratch[8];                               // stage events of ml_sig
    bool ev_scratch_valid = false;
    cudaStream_t side2 = nullptr;                            // small batches: [r_i] pk_i beside both the hash and the signature work
    cudaStream_t side = nullptr;                             // the signature-side MSM runs beside the per-set stages
    cudaStream_t chain = nullptr;                            // the RLC scalar chain (high priority, one SM-sized block)
    bool use_side = true;
    float stage_ms[ST_COUNT];
    int launches = 0;
    msm_state msm;
    // warp-cooperative dataflow programs (fpprog.hpp), compiled on first use and kept on the device
    struct dev_prog { uint32_t *d = nullptr; int nslots = 0, nrounds = 0, version = 1; };
    std::map<std::pair<int, int>, dev_prog> progs;           // keyed by (prog_kind, key)
    fp *d_small = nullptr;                                   // per-set program inputs/outputs of the small-batch route
    fp *d_norm = nullptr;                                    // [0] Fp norm taken out of the final exponentiation, [1] its inverse
    fp *d_consts = nullptr;                                  // Frobenius coefficients (fpprog::CONST_*)
    fp12 *d_gt = nullptr;                                    // final exponentiation result, Montgomery form
    fp12 *d_fold = nullptr;                                  // levels of the product of many partials (fold_partials)
    size_t fold_cap = 0;
    bool serial_tail = false;
    bool prog_smem_raised = false;                           // k_fp_program allowed > 48 KiB of shared memory on this device
    // host-buffer calls on large batches: the H2D copy is cut into H2D_SLICES pieces on a copy stream and the hash kernel
    // into as many launches on their own streams, each waiting for its piece only (run_partial_impl); created on first
    // use by create_slices
    const uint8_t *h_src = nullptr;                          // caller's host buffer for the current call (borrowed)
    cudaStream_t copy_stream = nullptr, slice_stream[H2D_SLICES] = {};
    cudaEvent_t ev_copy[H2D_SLICES] = {}, ev_slice[H2D_SLICES] = {};
    bool chain_smem_raised = false;                          // k_rlc_scalars allowed to reserve a whole SM's shared memory
    // multi-device context (blsgpu_create_multi): this context is the leader (share 0 + the one final exponentiation),
    // peers[k-1] owns share k on its own device; the 576-byte partials and the flags are gathered into the leader
    std::vector<blsgpu_ctx *> peers;
    fp12 *d_gather = nullptr;                                // ndev partials, share order
    int *d_gather_flags = nullptr;                           // ndev infinite-public-key flags
    cudaEvent_t ev_share = nullptr;                          // "this share's partial is ready" (recorded on the share's stream)
    size_t multi_cap = 0;                                    // capacity of the whole multi-device context (leader only)
    // CUDA graphs for the small-batch route: a block-sized batch is ~35 launches on three streams, i.e. ~40 driver calls
    // per batch from the host thread; the second call with the same (sets pointer, n, chunks) captures the whole
    // sequence (fork / join included) and every later one replays it with ONE launch.  The 32 random bytes reach the
    // scalar kernel through device memory (d_srb), refreshed by a copy node from a fixed pinned address.
    struct graph_entry { const void *sets; size_t n; uint32_t chunks; int seen; cudaGraphExec_t exec; };
    std::vector<graph_entry> graphs;
    bool use_graph = true;
    bool srb_from_dev = false;                               // launch_scalars: read the random bytes from d_srb
    uint32_t *d_srb = nullptr;
    std::string err;
};

static thread_local std::string g_err;                   // blsgpu_create failures, read back by the calling thread

static int fail(blsgpu_ctx *c, int code, const char *what, cudaError_t e = cudaSuccess) {
    char buf[512];
    if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(buf, sizeof buf, "%s", what);
    if (c) c->err = buf; else g_err = buf;
    return code;
}

#define CK(call)                                                                  \
    do {                                                                          \
        cudaError_t e_ = (call);                                                  \
        if (e_ != cudaSuccess) return fail(ctx, BLSGPU_ERR_CUDA, #call, e_);      \
    } while (0)

static inline unsigned nblk(size_t n, unsigned bs = 128) { return (unsigned)((n + bs - 1) / bs); }

// the route thresholds, read from the environment once per process (route.hpp)
static const route::thresholds &thr() {
    static const route::thresholds t = route::read_thresholds();
    return t;
}

extern "C" int blsgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" const char *blsgpu_last_error(const blsgpu_ctx *ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }
extern "C" size_t blsgpu_capacity(const blsgpu_ctx *ctx) { return ctx ? (ctx->multi_cap ? ctx->multi_cap : ctx->cap) : 0; }

static void destroy_slices(blsgpu_ctx *ctx) {
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    ctx->copy_stream = nullptr;
    for (int k = 0; k < H2D_SLICES; k++) {
        if (ctx->slice_stream[k]) cudaStreamDestroy(ctx->slice_stream[k]);
        if (ctx->ev_copy[k]) cudaEventDestroy(ctx->ev_copy[k]);
        if (ctx->ev_slice[k]) cudaEventDestroy(ctx->ev_slice[k]);
        ctx->slice_stream[k] = nullptr;
        ctx->ev_copy[k] = ctx->ev_slice[k] = nullptr;
    }
}

// the copy stream and the streams and events of the slices; all or none: on failure the context is left without them
static cudaError_t create_slices(blsgpu_ctx *ctx) {
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    for (int k = 0; k < H2D_SLICES && e == cudaSuccess; k++) {
        e = cudaStreamCreateWithFlags(&ctx->slice_stream[k], cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_copy[k], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_slice[k], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) destroy_slices(ctx);
    return e;
}

extern "C" void blsgpu_destroy(blsgpu_ctx *ctx) {
    if (!ctx) return;
    for (blsgpu_ctx *p : ctx->peers) blsgpu_destroy(p);
    ctx->peers.clear();
    cudaSetDevice(ctx->device);
    cudaFree(ctx->d_gather); cudaFree(ctx->d_gather_flags); cudaFree(ctx->d_srb);
    miller_ws_free(ctx->ml);
    miller_ws_free(ctx->ml_sig);
    for (auto &g : ctx->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    if (ctx->ev_share) cudaEventDestroy(ctx->ev_share);
    destroy_slices(ctx);
    if (ctx->ev_scratch_valid) for (int i = 0; i < 8; i++) cudaEventDestroy(ctx->ev_scratch[i]);
    cudaFree(ctx->d_sets); cudaFree(ctx->d_r); cudaFree(ctx->d_H); cudaFree(ctx->d_Pj); cudaFree(ctx->d_Q);
    cudaFree(ctx->d_P); cudaFree(ctx->d_S); cudaFree(ctx->d_partials); cudaFree(ctx->d_gtb);
    cudaFree(ctx->d_flags); cudaFree(ctx->d_dbg); cudaFree(ctx->d_misc); cudaFree(ctx->d_misc2); cudaFree(ctx->d_consts); cudaFree(ctx->d_gt);
    for (auto &kv : ctx->progs) cudaFree(kv.second.d);
    cudaFree(ctx->d_norm); cudaFree(ctx->d_small); cudaFree(ctx->d_fold);
    msm_free(ctx->msm);
    if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
    for (int i = 0; i < 2 * ST_COUNT + 5; i++) if (ctx->ev_valid[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->side) cudaStreamDestroy(ctx->side);
    if (ctx->chain) cudaStreamDestroy(ctx->chain);
    if (ctx->side2) cudaStreamDestroy(ctx->side2);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

extern "C" blsgpu_ctx *blsgpu_create(int device, size_t max_sets) {
    int ndev = blsgpu_device_count();
    if (ndev <= 0) { fail(nullptr, 0, "blsgpu_create: no CUDA device (this library has no CPU path)"); return nullptr; }
    if (device < 0 || device >= ndev) { fail(nullptr, 0, "blsgpu_create: bad device index"); return nullptr; }
    if (max_sets == 0) max_sets = 1;
    blsgpu_ctx *ctx = new blsgpu_ctx();
    ctx->device = device;
    ctx->cap = max_sets;
    for (int i = 0; i < 2 * ST_COUNT + 5; i++) ctx->ev_valid[i] = false;
    for (int i = 0; i < ST_COUNT; i++) ctx->stage_ms[i] = 0.f;
    cudaError_t e = cudaSetDevice(device);
    auto bad = [&](const char *what, cudaError_t err) {
        fail(nullptr, 0, what, err);
        blsgpu_destroy(ctx);
        return (blsgpu_ctx *)nullptr;
    };
    if (e != cudaSuccess) return bad("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bad("cudaStreamCreate", e);
    ctx->stream = ctx->ml.stream = ctx->own_stream;
    { int sms = 0; if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) ctx->msm.sms = sms; }
    size_t n = max_sets;
#define ALLOC(ptr, bytes) if ((e = cudaMalloc((void **)&(ptr), (bytes))) != cudaSuccess) return bad("cudaMalloc " #ptr, e)
    ALLOC(ctx->d_sets, n * sizeof(sigset));
    ALLOC(ctx->d_r, n * 8);
    ALLOC(ctx->d_H, n * sizeof(g2_jac));
    ALLOC(ctx->d_Pj, n * sizeof(g1_jac));
    ALLOC(ctx->d_Q, (n + 1) * sizeof(g2_aff));            // + the signature-side pair
    ALLOC(ctx->d_P, (n + 1) * sizeof(g1_aff));
    ALLOC(ctx->d_S, n * sizeof(g2_jac));
    ctx->ml.caps = route::miller_caps_batch(thr(), n);
    if ((e = miller_ws_alloc(ctx->ml)) != cudaSuccess) return bad("cudaMalloc Miller workspace", e);
    ctx->ml.ev = ctx->ev + 2 * ST_LINES;
    ALLOC(ctx->d_partials, 64 * sizeof(fp12));
    ALLOC(ctx->d_gtb, 576);
    ALLOC(ctx->d_gt, sizeof(fp12));
    ALLOC(ctx->d_consts, fpprog::CONST_COUNT * sizeof(fp));
    ALLOC(ctx->d_norm, 2 * sizeof(fp));
    ALLOC(ctx->d_flags, 4 * sizeof(int));
    if (getenv("BLSGPU_DEBUG_CHAIN")) ALLOC(ctx->d_dbg, 8 * sizeof(unsigned long long));
    ALLOC(ctx->d_srb, 32);
#undef ALLOC
    if ((e = cudaMallocHost((void **)&ctx->h_pinned, 4096)) != cudaSuccess) return bad("cudaMallocHost", e);
    // the programs' constant table, filled by a kernel from the __constant__ tables (a device-to-device
    // cudaMemcpyFromSymbol does the same, but compute-sanitizer's initcheck does not see constant memory as initialised)
    k_fill_consts<<<1, 64>>>(ctx->d_consts);
    if ((e = cudaGetLastError()) != cudaSuccess) return bad("k_fill_consts", e);
    if ((e = cudaDeviceSynchronize()) != cudaSuccess) return bad("cudaDeviceSynchronize", e);
    ctx->serial_tail = getenv("BLSGPU_SERIAL_TAIL") && atoi(getenv("BLSGPU_SERIAL_TAIL")) != 0;
    if (getenv("BLSGPU_ACC_TEAM")) ctx->acc_team = atoi(getenv("BLSGPU_ACC_TEAM")) != 0;
    for (int i = 0; i < 2 * ST_COUNT + 5; i++) {
        if ((e = cudaEventCreate(&ctx->ev[i])) != cudaSuccess) return bad("cudaEventCreate", e);
        ctx->ev_valid[i] = true;
    }
    // The scalar chain (ONE block that needs a whole SM to itself) has a stream of its own at the highest priority: when it
    // becomes runnable together with a grid that fills the machine (the hash kernel behind a caller's H2D copy on the main
    // stream) its block is placed first.  The signature-side sum that follows it stays at normal priority — at high
    // priority its grids push the hash kernel's blocks back and the step gets 3 % longer (measured).
    int pri_lo = 0, pri_hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&pri_lo, &pri_hi) != cudaSuccess) { cudaGetLastError(); pri_hi = 0; }
    if ((e = cudaStreamCreateWithPriority(&ctx->chain, cudaStreamNonBlocking, pri_hi)) != cudaSuccess) return bad("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking)) != cudaSuccess) return bad("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->side2, cudaStreamNonBlocking)) != cudaSuccess) return bad("cudaStreamCreate", e);
    if (getenv("BLSGPU_SIDE_STREAM")) ctx->use_side = atoi(getenv("BLSGPU_SIDE_STREAM")) != 0;
    if (getenv("BLSGPU_GRAPH")) ctx->use_graph = atoi(getenv("BLSGPU_GRAPH")) != 0;
    if ((e = cudaEventCreateWithFlags(&ctx->ev_share, cudaEventDisableTiming)) != cudaSuccess) return bad("cudaEventCreate", e);
    for (int i = 0; i < 8; i++) if ((e = cudaEventCreate(&ctx->ev_scratch[i])) != cudaSuccess) return bad("cudaEventCreate", e);
    ctx->ev_scratch_valid = true;
    ctx->ml_sig.caps = route::miller_caps_sig();
    ctx->ml_sig.stream = ctx->side;
    ctx->ml_sig.ev = ctx->ev_scratch;
    return ctx;
}

// Multi-GPU behind the ABI (SURVEY.md section 8b/8e): the fan-out that bls_batch_verifier.nim:316-369 does over Taskpools
// threads happens over devices inside the call.  devices[0] hosts the leader (share 0, the gather target and the one
// final exponentiation); a device index may be listed more than once (several shares on one GPU: the test boxes have one).
extern "C" blsgpu_ctx *blsgpu_create_multi(const int *devices, int ndev, size_t max_sets) {
    if (!devices || ndev <= 0 || ndev > 64) { fail(nullptr, 0, "blsgpu_create_multi: 1..64 devices"); return nullptr; }
    if (max_sets == 0) max_sets = 1;
    const size_t share = (max_sets + (size_t)ndev - 1) / (size_t)ndev;
    blsgpu_ctx *lead = blsgpu_create(devices[0], ndev == 1 ? max_sets : share);
    if (!lead) return nullptr;
    for (int k = 1; k < ndev; k++) {
        blsgpu_ctx *p = blsgpu_create(devices[k], share);
        if (!p) { blsgpu_destroy(lead); return nullptr; }           // g_err holds the reason
        lead->peers.push_back(p);
    }
    cudaError_t e = cudaSetDevice(lead->device);
    if (e == cudaSuccess) e = cudaMalloc((void **)&lead->d_gather, (size_t)ndev * sizeof(fp12));
    if (e == cudaSuccess) e = cudaMalloc((void **)&lead->d_gather_flags, (size_t)ndev * sizeof(int));
    if (e != cudaSuccess) { fail(nullptr, 0, "blsgpu_create_multi: gather buffers", e); blsgpu_destroy(lead); return nullptr; }
    // direct NVLink copies between the leader and every peer where the topology allows it (the 576-byte gather works
    // without it too: cudaMemcpyPeerAsync stages through the host then)
    for (blsgpu_ctx *p : lead->peers) {
        if (p->device == lead->device) continue;
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, lead->device, p->device) == cudaSuccess && can) {
            cudaSetDevice(lead->device);
            if (cudaDeviceEnablePeerAccess(p->device, 0) != cudaSuccess) cudaGetLastError();   // already enabled is fine
        }
    }
    cudaSetDevice(lead->device);
    lead->multi_cap = ndev == 1 ? max_sets : share * (size_t)ndev;
    return lead;
}
extern "C" int blsgpu_device_span(const blsgpu_ctx *ctx) { return ctx ? 1 + (int)ctx->peers.size() : 0; }

extern "C" int blsgpu_set_stream(blsgpu_ctx *ctx, void *cuda_stream) {
    if (!ctx) return BLSGPU_ERR_ARG;
    ctx->stream = ctx->ml.stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return 0;
}

static int ensure_misc(blsgpu_ctx *ctx, size_t bytes) {
    if (ctx->misc_bytes >= bytes) return 0;
    if (ctx->d_misc) cudaFree(ctx->d_misc);
    ctx->d_misc = nullptr;
    ctx->misc_bytes = 0;
    CK(cudaMalloc(&ctx->d_misc, bytes));
    ctx->misc_bytes = bytes;
    return 0;
}

static int ensure_misc2(blsgpu_ctx *ctx, size_t bytes) {
    if (ctx->d_misc2) return 0;
    CK(cudaMalloc(&ctx->d_misc2, bytes < 1024 ? 1024 : bytes));
    return 0;
}

static words8 words_of(const uint8_t b[32]) {
    words8 w;
    for (int i = 0; i < 8; i++)
        w.w[i] = ((uint32_t)b[4 * i] << 24) | ((uint32_t)b[4 * i + 1] << 16) | ((uint32_t)b[4 * i + 2] << 8) | b[4 * i + 3];
    return w;
}

#define BEGIN(stage, st) CK(cudaEventRecord(ctx->ev[2 * (stage)], st))
#define END(stage, st) CK(cudaEventRecord(ctx->ev[2 * (stage) + 1], st))
static_assert(fpprog::CONST_COUNT == fpprog_const_count && fpprog::CONST_FROB1 == 0 && fpprog::CONST_FROB2 == 10 &&
                  fpprog::CONST_FROB3 == 20 && fpprog::CONST_PSI_CX == 30 && fpprog::CONST_PSI_CY == 32 &&
                  fpprog::CONST_PSI2_CX == 34 && fpprog::CONST_ONE == 35, "k_fill_consts layout");
#define EV_FORK (2 * ST_COUNT)
#define EV_JOIN (2 * ST_COUNT + 1)
#define EV_G1 (2 * ST_COUNT + 2)
#define EV_SC (2 * ST_COUNT + 3)
#define EV_HASHED (2 * ST_COUNT + 4)

static route::batch_plan batch_plan_of(const blsgpu_ctx *ctx, size_t n, size_t total_n, uint32_t chunks, bool host_src, bool scalars) {
    return route::plan_batch(thr(), {ctx->use_side, ctx->acc_team, ctx->serial_tail, ctx->use_graph}, n, total_n, chunks, host_src,
                             scalars);
}

// scalars for global indices [first, first+n) into d_r; hog: the block of chains reserves an SM (route::chain_hog)
static int launch_scalars(blsgpu_ctx *ctx, const uint8_t srb[32], size_t n, size_t first, size_t total_n,
                          uint32_t chunks, const uint64_t *scalars, bool hog, cudaStream_t s) {
    if (scalars) {
        for (size_t i = 0; i < n; i++) if (scalars[i] == 0) return fail(ctx, BLSGPU_ERR_ARG, "explicit RLC scalar is zero");
        CK(cudaMemcpyAsync(ctx->d_r, scalars, n * 8, cudaMemcpyHostToDevice, s));
        return 0;
    }
    if (!srb) return fail(ctx, BLSGPU_ERR_ARG, "secureRandomBytes is NULL");
    const size_t nb = route::rlc_chains(total_n, chunks);
    const size_t smem = hog ? 227 * 1024 : 0;
    if (hog && !ctx->chain_smem_raised) {
        CK(cudaFuncSetAttribute(k_rlc_scalars, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctx->chain_smem_raised = true;
    }
    // d_flags[3]: "the block of chains is resident" (cleared with the other flags at the start of the call)
    volatile int *started = hog && ctx->use_side ? ctx->d_flags + 3 : nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)nblk(nb, 32));
    cfg.blockDim = dim3(32);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    const uint32_t *d_srb = nullptr;
    words8 w8 = words8();
    if (ctx->srb_from_dev) {
        // h_pinned + 1024: 8 big-endian words written by the caller of the captured sequence before every launch
        CK(cudaMemcpyAsync(ctx->d_srb, ctx->h_pinned + 1024, 32, cudaMemcpyHostToDevice, s));
        d_srb = ctx->d_srb;
    } else {
        w8 = words_of(srb);
    }
    CK(cudaLaunchKernelEx(&cfg, k_rlc_scalars, w8, d_srb, total_n, chunks, first, n, ctx->d_r, started, ctx->d_dbg));
    ctx->launches++;
    CK(cudaGetLastError());
    return 0;
}

enum { SETPROG_COFACTOR = 0, SETPROG_G2MUL64 = 1, SETPROG_LINES = 2 };

// Compile (once) and fetch a program:
//   PROG_COMBINE        combine over `key` segments
//   PROG_FINAL          final exponentiation of `key` partials with the Fp inversion supplied in IN1
//   PROG_NORM           the norm that inversion applies to (fpprog.hpp build_final)
//   PROG_SET            per-set G2 program `key` (SETPROG_*)
//   PROG_PRODUCT        product tree over `key` Fp12 values
//   PROG_MSM_HORNER_G*  window Horner of an MSM, key = nwin * 64 + c (c < 64)
// A first use uploads the program on stream st and waits for it.  A tail program that does not build fails the call;
// a Horner program that does not build or needs more than 48 KiB of shared memory is cached as absent (out.d == nullptr),
// and the MSM runs k_msm_horner instead.
static int get_prog(blsgpu_ctx *ctx, prog_kind kind, int key, blsgpu_ctx::dev_prog &out, cudaStream_t st) {
    auto it = ctx->progs.find({kind, key});
    if (it != ctx->progs.end()) { out = it->second; return 0; }
    fpprog::Program P;
    const bool horner = kind == PROG_MSM_HORNER_G1 || kind == PROG_MSM_HORNER_G2;
    if (kind == PROG_COMBINE) {
        int len[64];
        for (int j = 0; j < key; j++) len[j] = ml_seg_hi(j, key) - ml_seg_lo(j, key) + 1;
        P = fpprog::build_combine(key, len);
    } else if (kind == PROG_PRODUCT) {                   // product of `key` Fp12 values (GT product of a small batch)
        P = fpprog::build_fp12_product(key);
    } else if (kind == PROG_SET) {                       // per-set programs of the small-batch route
        P = key == SETPROG_COFACTOR ? fpprog::build_g2_clear_cofactor() : (key == SETPROG_G2MUL64 ? fpprog::build_g2_mul64() : fpprog::build_miller_lines());
    } else if (horner) {
        P = kind == PROG_MSM_HORNER_G1 ? fpprog::build_msm_horner_g1(key / 64, key % 64) : fpprog::build_msm_horner_g2(key / 64, key % 64);
    } else {
        P = fpprog::build_final(key, kind == PROG_FINAL ? fpprog::INV_EXTERNAL : fpprog::INV_EMIT_ARG);
    }
    blsgpu_ctx::dev_prog dp;
    if (horner && (!P.ok || (size_t)P.nslots * sizeof(fp) > 48 * 1024)) { ctx->progs[{kind, key}] = dp; out = dp; return 0; }
    if (!P.ok) return fail(ctx, BLSGPU_ERR_ARG, "tail program does not fit the slot file");
    dp.nslots = P.nslots;
    dp.nrounds = P.nrounds;
    dp.version = P.version;
    CK(cudaMalloc((void **)&dp.d, P.words.size() * 4));
    // stream-ordered upload, completed before the host vector goes away (first use only)
    CK(cudaMemcpyAsync(dp.d, P.words.data(), P.words.size() * 4, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    ctx->progs[{kind, key}] = dp;
    out = dp;
    return 0;
}

// one warp per instance: n instances of a program (format 1 or 2, fpprog.hpp) on stream st, strides in field elements
static void launch_prog_many(blsgpu_ctx *ctx, const blsgpu_ctx::dev_prog &p, cudaStream_t st, size_t n, const fp *in0, size_t s_in0,
                             const fp *in1, size_t s_in1, fp *out0, size_t s_out, bool stream_outputs = false) {
    const size_t smem = (size_t)p.nslots * sizeof(fp);
    auto k = p.version == 2 ? (stream_outputs ? k_fp_program2_stream : k_fp_program2) : (stream_outputs ? k_fp_program_stream : k_fp_program);
    k<<<(unsigned)n, 32, smem, st>>>(p.d, in0, in1, ctx->d_consts, out0, s_in0, s_in1, s_out);
    ctx->launches++;
}

// one warp per (row, group of m columns): rows of `in` (stride in_stride Fp12) -> rows of `out` (stride out_stride)
static void launch_prog_rows(blsgpu_ctx *ctx, const blsgpu_ctx::dev_prog &p, cudaStream_t st, size_t blocks, const fp12 *in,
                             fp12 *out, unsigned m, size_t in_stride, size_t out_stride) {
    auto k = p.version == 2 ? k_fp_program2_rows : k_fp_program_rows;
    k<<<(unsigned)blocks, 32, (size_t)p.nslots * sizeof(fp), st>>>(p.d, (const fp *)in, ctx->d_consts, (fp *)out, m, in_stride, out_stride);
    ctx->launches++;
}

// one instance, which may use up to 64 KiB of shared memory
static int launch_prog(blsgpu_ctx *ctx, const blsgpu_ctx::dev_prog &p, cudaStream_t st, const fp *in0, fp *out0, const fp *in1 = nullptr) {
    if ((size_t)p.nslots * sizeof(fp) > 48 * 1024 && !ctx->prog_smem_raised) {
        // per context, not per process: the attribute belongs to the function on ONE device
        CK(cudaFuncSetAttribute(k_fp_program, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        CK(cudaFuncSetAttribute(k_fp_program2, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        ctx->prog_smem_raised = true;
    }
    launch_prog_many(ctx, p, st, 1, in0, 0, in1, 0, out0, 0);
    return 0;
}

// sum_i [k_i] P_i on stream s (msm.cuh msm_run) in the shape route::plan_msm picks, the window Horner as a program when
// the plan allows it and the program builds; a failure is reported into ctx
template <class F>
static int run_msm(blsgpu_ctx *ctx, const uint8_t *d_points, size_t pstride, const uint8_t *d_scalars, size_t sstride, size_t n,
                   int nbits, cudaStream_t s, jac_t<F> *d_out_jac, aff_t<F> *d_out_aff) {
    const route::msm_plan p = route::plan_msm(thr(), n, nbits, ctx->msm.sms);
    blsgpu_ctx::dev_prog hp;
    if (p.horner_prog) {
        int rc = get_prog(ctx, std::is_same<F, fp>::value ? PROG_MSM_HORNER_G1 : PROG_MSM_HORNER_G2, p.nwin * 64 + p.c, hp, s);
        if (rc) return rc;
    }
    std::function<void(cudaStream_t, const fp *, fp *)> horner;
    if (hp.d) horner = [&](cudaStream_t ts, const fp *in, fp *out) { launch_prog_many(ctx, hp, ts, 1, in, 0, nullptr, 0, out, 0); };
    std::string err;
    int rc = msm_run<F>(ctx->msm, p, horner, d_points, pstride, d_scalars, sstride, n, nbits, s, d_out_jac, d_out_aff,
                        &ctx->launches, err);
    return rc ? fail(ctx, rc == -1 ? BLSGPU_ERR_CUDA : BLSGPU_ERR_ARG, err.c_str()) : 0;
}

// Per-set inputs and outputs of the small-batch route's programs, SMALL_ROUTE_CAP sets each: homogeneous points of 6
// field elements, and the 64 bits of a scalar as field elements 0 / 1
struct small_bufs { fp *hash_in, *hash_out, *sig_in, *sig_out, *bits; };

// the small-route buffers, allocated on first use
static int small_buffers(blsgpu_ctx *ctx, small_bufs &b) {
    const size_t cap = route::SMALL_ROUTE_CAP;
    if (!ctx->d_small) CK(cudaMalloc((void **)&ctx->d_small, cap * (6 + 6 + 6 + 6 + 64) * sizeof(fp)));
    b.hash_in = ctx->d_small;
    b.hash_out = b.hash_in + 6 * cap;
    b.sig_in = b.hash_out + 6 * cap;
    b.sig_out = b.sig_in + 6 * cap;
    b.bits = b.sig_out + 6 * cap;
    return 0;
}

// H(m_i) of the small-batch route on stream s, up to the homogeneous point in b.hash_out: the map to E2 (two lanes per
// message, or the pair kernel with BLSGPU_MAP_LANES2=0) into b.hash_in, then the cofactor clearing as a per-set program.
// The messages are those of `sets`, or with sets == nullptr msgs + offs[i] .. offs[i + 1] under the tag dst.
static int launch_small_hash(blsgpu_ctx *ctx, const small_bufs &b, cudaStream_t s, size_t n, const sigset *sets,
                             const uint8_t *msgs, const uint32_t *offs, const uint8_t *dst, size_t dst_len) {
    blsgpu_ctx::dev_prog p_cof;
    int rc = get_prog(ctx, PROG_SET, SETPROG_COFACTOR, p_cof, s);
    if (rc) return rc;
    if (thr().map_lanes2) k_hash_map_lanes2<<<nblk(2 * n, 64), 64, 0, s>>>(sets, msgs, offs, dst, (uint32_t)dst_len, n, b.hash_in);
    else if (sets) k_hash_map_pair<<<nblk(2 * n), 128, 0, s>>>(sets, n, b.hash_in);
    else k_hash_map_pair_msgs<<<nblk(2 * n), 128, 0, s>>>(msgs, offs, dst, (uint32_t)dst_len, n, b.hash_in);
    launch_prog_many(ctx, p_cof, s, n, b.hash_in, 6, nullptr, 0, b.hash_out, 6);
    return 0;
}

// Multi-Miller loop over the np pairs (d_Q[pair0 + i], d_P[pair0 + i]) + reductions, on the buffers, stream and stage
// events of workspace ws; leaves conj(prod ML) in d_partials[slot]
static int run_miller(blsgpu_ctx *ctx, miller_ws &ws, size_t np, int slot, size_t pair0 = 0) {
#define WBEGIN(stage) CK(cudaEventRecord(ws.ev[2 * ((stage) - ST_LINES)], s))
#define WEND(stage) CK(cudaEventRecord(ws.ev[2 * ((stage) - ST_LINES) + 1], s))
    cudaStream_t s = ws.stream;
    int rc;
    // tile by tile: lines, then per-(group, segment) accumulation
    const bool team = ctx->acc_team;
    const size_t lines_cap = ws.caps.lines_cap;
    const route::miller_plan mp = route::plan_miller(thr(), np, lines_cap, team, ctx->serial_tail);
    const int G = mp.G, nseg = mp.nseg;
    const size_t ncols = mp.ncols, row_stride = mp.row_stride, ncols2 = mp.ncols2;
    // every default plan fits (tests/test_hostsim.py); threshold overrides may not
    if (!route::fits(mp, ws.caps)) return fail(ctx, BLSGPU_ERR_CAPACITY, "segment product buffer too small");
    size_t col = 0;
    WBEGIN(ST_LINES);
    bool single = np <= lines_cap;
    for (size_t off = 0; off < np; off += lines_cap) {
        size_t t = np - off < lines_cap ? np - off : lines_cap;
        size_t stride = lines_cap;
        const int lines = off + t < np ? mp.lines : mp.lines_last;
        if (lines == route::LINES_PROGRAM) {
            // one warp per pair runs the 68 line evaluations as a dataflow program, then a scatter into the
            // accumulation's layout
            blsgpu_ctx::dev_prog lp;
            rc = get_prog(ctx, PROG_SET, SETPROG_LINES, lp, s);
            if (rc) return rc;
            const size_t per = (size_t)ML_NLINES * 6;
            if (!ws.small_lines) CK(cudaMalloc((void **)&ws.small_lines, ws.caps.small_lines * per * sizeof(fp)));
            launch_prog_many(ctx, lp, s, t, (const fp *)(ctx->d_Q + pair0), 4, (const fp *)(ctx->d_P + pair0), 2, ws.small_lines, per, true);
            k_lines_from_prog<<<nblk(t * ML_NLINES * ML_LINE_WORDS, 256), 256, 0, s>>>((const uint32_t *)ws.small_lines, ctx->d_Q + pair0, ctx->d_P + pair0, t,
                                                                                      ws.lines, stride);
            ctx->launches++;
        } else if (lines == route::LINES_LANES2) {
            k_miller_lines_lanes2<<<nblk(2 * t), 128, 0, s>>>(ctx->d_Q + pair0 + off, ctx->d_P + pair0 + off, t, ws.lines, stride);
        } else {
            k_miller_lines<<<nblk(t), 128, 0, s>>>(ctx->d_Q + pair0 + off, ctx->d_P + pair0 + off, t, ws.lines, stride);
        }
        if (single) { WEND(ST_LINES); WBEGIN(ST_ACC); }
        size_t ngroups = (t + G - 1) / G;
        if (team) {
            dim3 grid(nblk(ngroups, ACC_TPB), nseg);
            k_miller_acc_team<<<grid, ACC_BS, 0, s>>>(ws.lines, stride, t, ngroups, G, nseg, ws.F, row_stride, col);
            col += ngroups;
        } else {
            dim3 grid(nblk(ngroups, BLS_ACC_BS), nseg);
            k_miller_acc<<<grid, BLS_ACC_BS, 0, s>>>(ws.lines, stride, t, ngroups, G, nseg, ws.F, ncols, col);
            col += grid.x;
        }
        ctx->launches += 2;
    }
    if (!single) { WEND(ST_LINES); WBEGIN(ST_ACC); }        // multi-tile: lines+acc are reported together under miller_lines
    WEND(ST_ACC);
    WBEGIN(ST_GTPROD);
    if (ncols == 1) {                                       // one group: the segment values are the products already
        CK(cudaMemcpy2DAsync(ws.seg, sizeof(fp12), ws.F, row_stride * sizeof(fp12), sizeof(fp12), (size_t)nseg,
                             cudaMemcpyDeviceToDevice, s));
    } else if (mp.gt_prog) {
        // product trees of eight as dataflow programs, one warp per (segment row, group of 8 columns), level after level
        // (the 54 multiplications of a tree node spread over the 32 lanes); the rows ping-pong between F and F2 and
        // every level's rows are padded with ones to a multiple of 8
        blsgpu_ctx::dev_prog p8, pm;
        fp12 *cur = ws.F, *other = ws.F2;
        size_t cols = ncols, stride = row_stride;
        while (cols > 8) {
            const size_t m = (cols + 7) / 8, m_stride = m > 8 ? ((m + 7) & ~(size_t)7) : m;
            rc = get_prog(ctx, PROG_PRODUCT, 8, p8, s);
            if (rc) return rc;
            if (cols & 7) { k_fp12_pad_one<<<nseg, 32, 0, s>>>(cur, stride, cols); ctx->launches++; }
            launch_prog_rows(ctx, p8, s, (size_t)nseg * m, cur, other, (unsigned)m, stride, m_stride);
            fp12 *t = cur; cur = other; other = t;
            cols = m;
            stride = m_stride;
        }
        rc = get_prog(ctx, PROG_PRODUCT, (int)cols, pm, s);
        if (rc) return rc;
        launch_prog_rows(ctx, pm, s, (size_t)nseg, cur, ws.seg, 1u, stride, 1);
    } else if (ncols > BLS_ACC_BS) {
        dim3 grid((unsigned)ncols2, nseg);
        k_fp12_rows_step<<<grid, BLS_ACC_BS, 0, s>>>(ws.F, ncols, ncols, ws.F2, ncols2);
        k_fp12_rows<<<nseg, BLS_ACC_BS, 0, s>>>(ws.F2, ncols2, ncols2, ws.seg);
        ctx->launches++;
    } else {
        k_fp12_rows<<<nseg, BLS_ACC_BS, 0, s>>>(ws.F, ncols, ncols, ws.seg);
    }
    WEND(ST_GTPROD);
    WBEGIN(ST_PARTIAL);
    ctx->launches++;
    if (ctx->serial_tail) {
        k_combine<<<1, 32, 0, s>>>(ws.seg, nseg, ctx->d_partials + slot);
        ctx->launches++;
    } else {
        blsgpu_ctx::dev_prog cp;
        rc = get_prog(ctx, PROG_COMBINE, nseg, cp, s);
        if (rc) return rc;
        rc = launch_prog(ctx, cp, s, (const fp *)ws.seg, (fp *)(ctx->d_partials + slot));
        if (rc) return rc;
    }
    WEND(ST_PARTIAL);
    CK(cudaGetLastError());
    return 0;
#undef WBEGIN
#undef WEND
}

static int run_partial_impl(blsgpu_ctx *ctx, const sigset *d_sets, size_t n, size_t first, size_t total_n,
                            const uint8_t srb[32], uint32_t chunks, const uint64_t *scalars, int slot);
// all per-set stages + reductions; leaves the rank partial in d_partials[slot].  On failure nothing queued by the call
// is left in flight (the side streams were forked off and the caller may free its buffers right after the error).
static int run_partial(blsgpu_ctx *ctx, const sigset *d_sets, size_t n, size_t first, size_t total_n,
                       const uint8_t srb[32], uint32_t chunks, const uint64_t *scalars, int slot) {
    int rc = run_partial_impl(ctx, d_sets, n, first, total_n, srb, chunks, scalars, slot);
    if (rc) {
        cudaStreamSynchronize(ctx->chain);
        cudaStreamSynchronize(ctx->side);
        cudaStreamSynchronize(ctx->side2);
        if (ctx->copy_stream) {
            cudaStreamSynchronize(ctx->copy_stream);
            for (int k = 0; k < H2D_SLICES; k++) cudaStreamSynchronize(ctx->slice_stream[k]);
        }
        cudaStreamSynchronize(ctx->stream);
        cudaGetLastError();
    }
    if (!rc && ctx->d_dbg) {                                  // BLSGPU_DEBUG_CHAIN: when did the chain block start / end
        unsigned long long h[8];
        cudaStreamSynchronize(ctx->chain);
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(h, ctx->d_dbg, sizeof(h), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[blsgpu chain] n=%zu start->end %.3f ms, wait exit - chain start %.3f ms, sm %llu, seen %llu\n", n,
                (double)(h[1] - h[0]) * 1e-6, ((double)h[2] - (double)h[0]) * 1e-6, h[3], h[4]);
    }
    return rc;
}
static int run_partial_impl(blsgpu_ctx *ctx, const sigset *d_sets, size_t n, size_t first, size_t total_n,
                            const uint8_t srb[32], uint32_t chunks, const uint64_t *scalars, int slot) {
    cudaStream_t s = ctx->stream;
    ctx->launches = 0;
    if (!scalars && !srb) return fail(ctx, BLSGPU_ERR_ARG, "secureRandomBytes is NULL");
    const route::batch_plan plan = batch_plan_of(ctx, n, total_n, chunks, ctx->h_src != nullptr, scalars != nullptr);
    // Host-buffer call (blsgpu_batch_verify): this function issues the H2D copy itself.  Small and mid-size batches: one
    // copy ahead of everything.  Large ones: H2D_SLICES pieces on a copy stream, each followed at once by the launch of
    // the hash kernel over that piece on its own stream, so the copy (and, for pageable memory, the host-side staging
    // that blocks the calling thread piece by piece) hides behind H(m_i) of the earlier pieces.
    const bool sliced = plan.sliced;
    if (ctx->h_src && !sliced) CK(cudaMemcpyAsync(ctx->d_sets, ctx->h_src, n * sizeof(sigset), cudaMemcpyHostToDevice, s));
    if (sliced && !ctx->copy_stream) CK(create_slices(ctx));
    CK(cudaMemsetAsync(ctx->d_flags, 0, 4 * sizeof(int), s));
    // fork: the scalar chain (strictly sequential SHA-256 per reference chunk: tens of milliseconds for a large batch
    // when the caller passes tp.numThreads = 16..32 chunks) and the signature-side sum that consumes the scalars run on
    // a second stream, beside H(m_i), which needs neither; [r_i]pk_i waits for the scalars, the Miller loop for the sum
    cudaStream_t g = ctx->use_side ? ctx->side : s, cs = ctx->use_side ? ctx->chain : s;
    if (ctx->use_side) {
        CK(cudaEventRecord(ctx->ev[EV_FORK], s));
        CK(cudaStreamWaitEvent(cs, ctx->ev[EV_FORK], 0));
        CK(cudaStreamWaitEvent(g, ctx->ev[EV_FORK], 0));
    }
    BEGIN(ST_SCALARS, cs);
    int rc = launch_scalars(ctx, srb, n, first, total_n, chunks, scalars, plan.chain_hog, cs);
    if (rc) return rc;
    END(ST_SCALARS, cs);
    if (ctx->use_side) {
        CK(cudaEventRecord(ctx->ev[EV_SC], cs));
        CK(cudaStreamWaitEvent(g, ctx->ev[EV_SC], 0));
    }
    if (plan.chain_wait) {
        // the main stream (whose next kernel fills the machine) waits until the chains' block is placed: ~10 us when the
        // device is idle, at most 0.2 ms (400 000 cycles) when it is not
        k_wait_started<<<1, 32, 0, s>>>(ctx->d_flags + 3, 400000, ctx->d_dbg);
        ctx->launches++;
    }
    // Small-batch route: the serial stretches of a set (cofactor clearing, [r_i] sig_i) run as per-set dataflow
    // programs, one warp per set (fpprog.hpp build_g2_clear_cofactor / build_g2_mul64)
    blsgpu_ctx::dev_prog p_mul;
    small_bufs sb = {};
    if (plan.small) {
        rc = small_buffers(ctx, sb);
        if (!rc) rc = get_prog(ctx, PROG_SET, SETPROG_G2MUL64, p_mul, s);
        if (rc) return rc;
    }
    if (sliced) {
        if (!ctx->use_side) CK(cudaEventRecord(ctx->ev[EV_FORK], s));
        BEGIN(ST_HASH, s);
        const size_t per = ((n + H2D_SLICES - 1) / H2D_SLICES + 127) & ~(size_t)127;      // whole thread blocks per piece
        for (int k = 0; k < H2D_SLICES; k++) {
            const size_t off = (size_t)k * per;
            if (off >= n) { CK(cudaEventRecord(ctx->ev_copy[k], ctx->copy_stream)); CK(cudaEventRecord(ctx->ev_slice[k], ctx->copy_stream)); continue; }
            const size_t len = n - off < per ? n - off : per;
            if (k == 0) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev[EV_FORK], 0));     // after whatever preceded on s
            CK(cudaMemcpyAsync(ctx->d_sets + off, ctx->h_src + off * sizeof(sigset), len * sizeof(sigset), cudaMemcpyHostToDevice,
                               ctx->copy_stream));
            CK(cudaEventRecord(ctx->ev_copy[k], ctx->copy_stream));
            cudaStream_t sk = ctx->slice_stream[k];
            CK(cudaStreamWaitEvent(sk, ctx->ev_copy[k], 0));
            if (plan.hash == route::HASH_LANES2) k_hash_sets_lanes2<<<nblk(2 * len), 128, 0, sk>>>(d_sets + off, len, ctx->d_H + off);
            else k_hash_sets<<<nblk(len), 128, 0, sk>>>(d_sets + off, len, ctx->d_H + off);
            ctx->launches++;
            CK(cudaEventRecord(ctx->ev_slice[k], sk));
        }
        for (int k = 0; k < H2D_SLICES; k++) CK(cudaStreamWaitEvent(s, ctx->ev_slice[k], 0));
        END(ST_HASH, s);
        CK(cudaStreamWaitEvent(g, ctx->ev_copy[H2D_SLICES - 1], 0));    // the signature-side MSM reads every set
    }
    if (plan.g1_aside) {
        cudaStream_t g1s = ctx->side2;
        CK(cudaStreamWaitEvent(g1s, ctx->ev[EV_SC], 0));
        if (sliced) CK(cudaStreamWaitEvent(g1s, ctx->ev_copy[H2D_SLICES - 1], 0));   // the keys of every slice are in place
        BEGIN(ST_G1MUL, g1s);
        k_g1_mul<<<nblk(n), 128, 0, g1s>>>(d_sets, ctx->d_r, n, ctx->d_Pj, ctx->d_flags);
        END(ST_G1MUL, g1s);
        CK(cudaEventRecord(ctx->ev[EV_G1], g1s));
    }
    // H(m_i) on the main stream (already launched piece by piece when the host copy is sliced)
    auto launch_hash = [&]() -> int {
        if (sliced) return 0;
        BEGIN(ST_HASH, s);
        if (plan.hash == route::HASH_PROGRAM) {
            int rch = launch_small_hash(ctx, sb, s, n, d_sets, nullptr, nullptr, nullptr, 0);
            if (rch) return rch;
            k_g2_hom_to_jac<<<nblk(n), 128, 0, s>>>(sb.hash_out, n, ctx->d_H);
            ctx->launches += 2;                             // the map and the conversion
        } else if (plan.hash == route::HASH_LANES2) k_hash_sets_lanes2<<<nblk(2 * n), 128, 0, s>>>(d_sets, n, ctx->d_H);
        else if (plan.hash == route::HASH_PAIR) k_hash_sets_pair<<<nblk(2 * n), 128, 0, s>>>(d_sets, n, ctx->d_H);
        else k_hash_sets<<<nblk(n), 128, 0, s>>>(d_sets, n, ctx->d_H);
        END(ST_HASH, s);
        return 0;
    };
    if (plan.msm_after_hash) {
        rc = launch_hash();
        if (rc) return rc;
        CK(cudaEventRecord(ctx->ev[EV_HASHED], s));
        CK(cudaStreamWaitEvent(g, ctx->ev[EV_HASHED], 0));
    }
    BEGIN(ST_G2MUL, g);
    // S = sum_i [r_i] sig_i
    if (plan.sig == route::SIG_MSM) {
        rc = run_msm<fp2>(ctx, (const uint8_t *)d_sets + offsetof(sigset, sig), sizeof(sigset), (const uint8_t *)ctx->d_r, 8, n, 64,
                          g, ctx->d_S, nullptr);
        if (rc) return rc;
        END(ST_G2MUL, g);
        BEGIN(ST_G2SUM, g);
    } else {
        if (plan.sig == route::SIG_PROGRAM) {
            k_g2_mul_prep<<<nblk(64 * n), 128, 0, g>>>(d_sets, ctx->d_r, n, sb.sig_in, sb.bits);
            launch_prog_many(ctx, p_mul, g, n, sb.sig_in, 6, sb.bits, 64, sb.sig_out, 6);
            k_g2_hom_to_jac<<<nblk(n), 128, 0, g>>>(sb.sig_out, n, ctx->d_S);
            ctx->launches += 2;
        } else {
            k_g2_mul<<<nblk(n), 128, 0, g>>>(d_sets, ctx->d_r, n, ctx->d_S);
            ctx->launches++;
        }
        END(ST_G2MUL, g);
        BEGIN(ST_G2SUM, g);
        for (size_t m = n; m > 1;) {
            size_t half = (m + 1) / 2;
            k_g2_tree<<<nblk(half), 128, 0, g>>>(ctx->d_S, m, half);
            ctx->launches++;
            m = half;
        }
    }
    k_sig_pair<<<1, 32, 0, g>>>(ctx->d_S, n, ctx->d_Q, ctx->d_P);
    ctx->launches++;
    END(ST_G2SUM, g);
    // Deferred signature pair: pair number n = (S, -G1) gets its own one-pair Miller loop right here on the side stream,
    // on its own workspace, beside the big loop of the main stream; after the join the two values are multiplied (one
    // Fp12 product program).  Same product of the same n + 1 Miller values, hence same GT.
    if (plan.defer_sig) {
        if (!ctx->ml_sig.lines) CK(miller_ws_alloc(ctx->ml_sig));
        rc = run_miller(ctx, ctx->ml_sig, 1, slot + 1, n);
        if (rc) return rc;
    }
    if (ctx->use_side) CK(cudaEventRecord(ctx->ev[EV_JOIN], g));
    if (!plan.msm_after_hash) {
        rc = launch_hash();
        if (rc) return rc;
    }
    if (plan.g1_aside) {
        CK(cudaStreamWaitEvent(s, ctx->ev[EV_G1], 0));
    } else {
        if (ctx->use_side) CK(cudaStreamWaitEvent(s, ctx->ev[EV_SC], 0));
        BEGIN(ST_G1MUL, s);
        k_g1_mul<<<nblk(n), 128, 0, s>>>(d_sets, ctx->d_r, n, ctx->d_Pj, ctx->d_flags);
        END(ST_G1MUL, s);
    }
    BEGIN(ST_AFFINE, s);
    if (plan.affine == route::AFFINE_BLOCK) {
        // one Euclid inversion per block of 128 threads, about 32 768 threads in flight: 1 set per thread up to 32 768
        // sets, up to AFF_B beyond
        int per = (int)((n + 32767) / 32768);
        if (per > AFF_B) per = AFF_B;
        k_pairs_affine<<<nblk((n + per - 1) / per), 128, 0, s>>>(ctx->d_H, ctx->d_Pj, n, ctx->d_Q, ctx->d_P, 2, 0, per);
    } else if (plan.affine == route::AFFINE_WARP) k_pairs_affine<<<(unsigned)n, 32, 0, s>>>(ctx->d_H, ctx->d_Pj, n, ctx->d_Q, ctx->d_P, 1, 1, AFF_B);
    else k_pairs_affine<<<nblk((n + AFF_B - 1) / AFF_B), 128, 0, s>>>(ctx->d_H, ctx->d_Pj, n, ctx->d_Q, ctx->d_P, 0, 0, AFF_B);
    END(ST_AFFINE, s);
    ctx->launches += 3;
    if (!plan.defer_sig) {
        if (ctx->use_side) CK(cudaStreamWaitEvent(s, ctx->ev[EV_JOIN], 0));   // join: pair number n is in place
        return run_miller(ctx, ctx->ml, n + 1, slot);
    }
    rc = run_miller(ctx, ctx->ml, n, slot);                  // the n set pairs; (S, -G1) is being done on the side stream
    if (rc) return rc;
    CK(cudaStreamWaitEvent(s, ctx->ev[EV_JOIN], 0));
    blsgpu_ctx::dev_prog p2;
    rc = get_prog(ctx, PROG_PRODUCT, 2, p2, s);
    if (rc) return rc;
    // in place: the program loads all 24 inputs into its slot file before the first round and stores at the end
    rc = launch_prog(ctx, p2, s, (const fp *)(ctx->d_partials + slot), (fp *)(ctx->d_partials + slot));
    if (rc) return rc;
    END(ST_PARTIAL, s);
    CK(cudaGetLastError());
    return 0;
}

// The final-exponentiation programs take at most FINAL_DIRECT_MAX partials: every partial holds 12 slots of the slot
// file from the first round on, and from 25 partials on the pair of programs no longer fits it.
static const int FINAL_DIRECT_MAX = 8;

// Multiply `count` > FINAL_DIRECT_MAX partials eight at a time (product programs, one warp per group), level after level,
// until at most FINAL_DIRECT_MAX remain; parts / count then name the last level.  The levels alternate between the two
// halves of ctx->d_fold.
static int fold_partials(blsgpu_ctx *ctx, cudaStream_t s, const fp12 *&parts, int &count) {
    const size_t half = ((size_t)count + 7) / 8;
    if (ctx->fold_cap < 2 * half) {
        cudaFree(ctx->d_fold);
        ctx->d_fold = nullptr;
        ctx->fold_cap = 0;
        CK(cudaMalloc((void **)&ctx->d_fold, 2 * half * sizeof(fp12)));
        ctx->fold_cap = 2 * half;
    }
    for (int level = 0; count > FINAL_DIRECT_MAX; level++) {
        fp12 *out = ctx->d_fold + (level & 1) * half;
        const int full = count / 8, rest = count % 8;
        blsgpu_ctx::dev_prog p8, pr;
        int rc = get_prog(ctx, PROG_PRODUCT, 8, p8, s);
        if (rc) return rc;
        launch_prog_many(ctx, p8, s, (size_t)full, (const fp *)parts, 8 * 12, nullptr, 0, (fp *)out, 12);
        if (rest > 1) {
            rc = get_prog(ctx, PROG_PRODUCT, rest, pr, s);
            if (rc) return rc;
            launch_prog_many(ctx, pr, s, 1, (const fp *)(parts + 8 * full), 0, nullptr, 0, (fp *)(out + full), 0);
        } else if (rest == 1) {
            CK(cudaMemcpyAsync(out + full, parts + 8 * full, sizeof(fp12), cudaMemcpyDeviceToDevice, s));
        }
        parts = out;
        count = full + (rest ? 1 : 0);
    }
    return 0;
}

// enqueue: product of the partials, final exponentiation, verdict + GT bytes, and their copies into h_pinned
static int run_final_enqueue(blsgpu_ctx *ctx, int count, const fp12 *d_partials = nullptr, const int *d_rank_flags = nullptr) {
    cudaStream_t s = ctx->stream;
    const fp12 *parts = d_partials ? d_partials : ctx->d_partials;
    BEGIN(ST_FINAL, s);
    if (ctx->serial_tail) {
        k_final<<<1, 32, 0, s>>>(parts, count, d_rank_flags, ctx->d_gtb, ctx->d_flags + 1);
        ctx->launches++;
    } else {
        // [fold ->] norm program -> one-thread binary-Euclid inversion -> main program (fpprog.hpp build_final)
        int nparts = count;
        if (nparts > FINAL_DIRECT_MAX) {
            int rc = fold_partials(ctx, s, parts, nparts);
            if (rc) return rc;
        }
        blsgpu_ctx::dev_prog fpn, fpg;
        int rc = get_prog(ctx, PROG_NORM, nparts, fpn, s);
        if (!rc) rc = get_prog(ctx, PROG_FINAL, nparts, fpg, s);
        if (rc) return rc;
        rc = launch_prog(ctx, fpn, s, (const fp *)parts, ctx->d_norm);
        if (rc) return rc;
        k_fp_inv_one<<<1, 32, 0, s>>>(ctx->d_norm, ctx->d_norm + 1);
        ctx->launches++;
        rc = launch_prog(ctx, fpg, s, (const fp *)parts, (fp *)ctx->d_gt, ctx->d_norm + 1);
        if (rc) return rc;
        k_final_out<<<1, 32, 0, s>>>(ctx->d_gt, count, d_rank_flags, ctx->d_gtb, ctx->d_flags + 1);
        ctx->launches++;
    }
    END(ST_FINAL, s);
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->d_gtb, 576, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(ctx->h_pinned + 576, ctx->d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
    return 0;
}
// wait and read the verdict
static int run_final_finish(blsgpu_ctx *ctx, uint8_t gt_out[576], int *pk_inf, bool rank_flags) {
    CK(cudaStreamSynchronize(ctx->stream));
    int flags[4];
    memcpy(flags, ctx->h_pinned + 576, sizeof flags);
    // the gathered per-share flags when the caller supplies them (finalize_dev), else this context's own flag from the
    // run_partial that preceded (batch_verify_dev); never both: d_flags[0] may be stale from an earlier, unrelated batch
    if (pk_inf) *pk_inf = rank_flags ? flags[2] : flags[0];
    if (gt_out) memcpy(gt_out, ctx->h_pinned, 576);
    return flags[1] ? 1 : 0;
}
static int run_final(blsgpu_ctx *ctx, int count, uint8_t gt_out[576], int *pk_inf, const fp12 *d_partials = nullptr,
                     const int *d_rank_flags = nullptr) {
    int rc = run_final_enqueue(ctx, count, d_partials, d_rank_flags);
    if (rc) return rc;
    return run_final_finish(ctx, gt_out, pk_inf, d_rank_flags != nullptr);
}

static void collect_stage_times(blsgpu_ctx *ctx, bool with_final) {
    for (int i = 0; i < ST_COUNT; i++) {
        float ms = 0.f;
        if (i == ST_FINAL && !with_final) { ctx->stage_ms[i] = 0.f; continue; }
        if (cudaEventElapsedTime(&ms, ctx->ev[2 * i], ctx->ev[2 * i + 1]) != cudaSuccess) { cudaGetLastError(); ms = 0.f; }
        ctx->stage_ms[i] = ms;
    }
}

extern "C" int blsgpu_rlc_scalars(blsgpu_ctx *ctx, const uint8_t srb[32], size_t n, uint32_t chunks, uint64_t *out) {
    if (!ctx || !out) return BLSGPU_ERR_ARG;
    if (n == 0) return 0;
    if (n > ctx->cap) return fail(ctx, BLSGPU_ERR_CAPACITY, "batch larger than context capacity");
    CK(cudaSetDevice(ctx->device));
    int rc = launch_scalars(ctx, srb, n, 0, n, chunks, nullptr, route::chain_hog(thr(), n, chunks), ctx->stream);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, ctx->d_r, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// Small and mid-size batches (<= 8 192 sets: 30-45 launches on up to four streams, where launch gaps are 2-5 % of the
// call) through a CUDA graph.  First call with a key: direct launches (all lazy allocations and program uploads
// happen there).  Second call: the same sequence under stream capture (the fork to the side streams and the joins are
// captured with it), instantiated and launched.  Later calls: one cudaGraphLaunch.  `done` = the work of this call is
// queued and the caller only has to wait for it; done == false (first sighting, or capture unsupported) = run directly.
static int verify_graphed(blsgpu_ctx *ctx, const void *d_sets, size_t n, const uint8_t srb[32], uint32_t chunks, bool &done) {
    done = false;
    blsgpu_ctx::graph_entry *e = nullptr;
    for (auto &g : ctx->graphs) if (g.sets == d_sets && g.n == n && g.chunks == chunks) { e = &g; break; }
    if (!e) {
        if (ctx->graphs.size() >= 16) {                      // bounded cache: drop the oldest entry
            if (ctx->graphs.front().exec) cudaGraphExecDestroy(ctx->graphs.front().exec);
            ctx->graphs.erase(ctx->graphs.begin());
        }
        ctx->graphs.push_back({d_sets, n, chunks, 1, nullptr});
        return 0;
    }
    const words8 w = words_of(srb);
    memcpy(ctx->h_pinned + 1024, w.w, 32);                   // no copy is in flight: every call on a context ends with a sync
    if (!e->exec) {
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            ctx->use_graph = false;
            return 0;
        }
        ctx->srb_from_dev = true;
        int rc = run_partial_impl(ctx, (const sigset *)d_sets, n, 0, n, srb, chunks, nullptr, 0);
        if (!rc) rc = run_final_enqueue(ctx, 1);
        ctx->srb_from_dev = false;
        cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
        if (rc || ce != cudaSuccess || !graph) {
            cudaGetLastError();
            if (graph) cudaGraphDestroy(graph);
            ctx->use_graph = false;                          // run directly from now on (and for this call)
            return 0;
        }
        ce = cudaGraphInstantiate(&e->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { cudaGetLastError(); e->exec = nullptr; ctx->use_graph = false; return 0; }
    }
    CK(cudaGraphLaunch(e->exec, ctx->stream));
    ctx->launches = 1;
    done = true;
    return 0;
}

extern "C" int blsgpu_batch_verify_dev(blsgpu_ctx *ctx, const void *d_sets, size_t n, const uint8_t srb[32],
                                       uint32_t chunks, const uint64_t *scalars, uint8_t gt_out[576]) {
    if (!ctx) return BLSGPU_ERR_ARG;
    if (gt_out) memset(gt_out, 0, 576);
    if (n == 0) return 0;                                   // bls_batch_verifier.nim:137, :312
    if (!d_sets) return fail(ctx, BLSGPU_ERR_ARG, "sets is NULL");
    if ((uintptr_t)d_sets & 15) return fail(ctx, BLSGPU_ERR_ARG, "device sets pointer must be 16-byte aligned (TMA staging)");
    if (n > ctx->cap) return fail(ctx, BLSGPU_ERR_CAPACITY, "batch larger than context capacity");
    CK(cudaSetDevice(ctx->device));
    int rc, pk_inf = 0;
    if (srb && batch_plan_of(ctx, n, n, chunks, false, scalars != nullptr).graph) {
        bool done = false;
        rc = verify_graphed(ctx, d_sets, n, srb, chunks, done);
        if (rc) return rc;
        if (done) {
            rc = run_final_finish(ctx, gt_out, &pk_inf, false);
            for (int i = 0; i < ST_COUNT; i++) ctx->stage_ms[i] = 0.f;     // no event timing inside a graph (BLSGPU_GRAPH=0)
            if (rc < 0) return rc;
            if (pk_inf) { if (gt_out) memset(gt_out, 0, 576); return 0; }
            return rc;
        }
    }
    rc = run_partial(ctx, (const sigset *)d_sets, n, 0, n, srb, chunks, scalars, 0);
    if (rc) return rc;
    rc = run_final(ctx, 1, gt_out, &pk_inf);
    collect_stage_times(ctx, true);
    if (rc < 0) return rc;
    if (pk_inf) { if (gt_out) memset(gt_out, 0, 576); return 0; }   // update() failed -> false (aggregate.c:296)
    return rc;
}

// balanced contiguous split, the rule of blscurve/parallel_chunks.nim:42-55 applied to devices
static void share_range(size_t total, size_t parts, size_t k, size_t &first, size_t &len) {
    const size_t base = total / parts, rem = total % parts;
    if (k < rem) { first = (base + 1) * k; len = base + 1; }
    else { first = base * k + rem; len = base; }
}

// One batch over every device of a multi-device context, inside ONE call: share k goes to device k (H2D from the
// caller's buffer on that device's stream), every device leaves its 576-byte partial + flag in its own memory, the
// leader's stream waits for each share's event and pulls them over NVLink (cudaMemcpyPeerAsync), then runs the one final
// exponentiation.  Scalars come from the GLOBAL (n, chunks) derivation, so verdict and GT equal the one-device result.
static int batch_verify_multi(blsgpu_ctx *lead, const uint8_t *sets, size_t n, const uint8_t srb[32], uint32_t chunks,
                              const uint64_t *scalars, uint8_t gt_out[576]) {
    blsgpu_ctx *ctx = lead;                                  // CK() reports into the leader
    std::vector<blsgpu_ctx *> all;
    all.push_back(lead);
    for (blsgpu_ctx *p : lead->peers) all.push_back(p);
    const size_t ndev = all.size();
    int rc = 0, total_launches = 0;
    size_t issued = 0;
    for (size_t k = 0; k < ndev && rc == 0; k++) {
        blsgpu_ctx *c = all[k];
        size_t first, len;
        share_range(n, ndev, k, first, len);
        cudaError_t e = cudaSetDevice(c->device);
        if (e != cudaSuccess) { rc = fail(lead, BLSGPU_ERR_CUDA, "cudaSetDevice", e); break; }
        issued = k + 1;
        if (len == 0) {                                      // more devices than sets: neutral partial
            k_partial_one<<<1, 32, 0, c->stream>>>(c->d_partials, c->d_flags);
            c->launches = 1;
        } else {
            e = cudaMemcpyAsync(c->d_sets, sets + first * sizeof(sigset), len * sizeof(sigset), cudaMemcpyHostToDevice, c->stream);
            if (e != cudaSuccess) { rc = fail(lead, BLSGPU_ERR_CUDA, "cudaMemcpyAsync(share)", e); break; }
            rc = run_partial(c, c->d_sets, len, first, n, srb, chunks, scalars ? scalars + first : nullptr, 0);
            if (rc && c != lead) lead->err = c->err;
        }
        total_launches += c->launches;
        if (rc == 0 && (e = cudaEventRecord(c->ev_share, c->stream)) != cudaSuccess) rc = fail(lead, BLSGPU_ERR_CUDA, "cudaEventRecord", e);
    }
    if (rc) {                                                // nothing of this call may outlive it: the caller owns `sets`
        for (size_t k = 0; k < issued; k++) { cudaSetDevice(all[k]->device); cudaStreamSynchronize(all[k]->stream); }
        cudaSetDevice(lead->device);
        return rc;
    }
    CK(cudaSetDevice(lead->device));
    for (size_t k = 0; k < ndev; k++) {
        blsgpu_ctx *c = all[k];
        CK(cudaStreamWaitEvent(lead->stream, c->ev_share, 0));
        CK(cudaMemcpyPeerAsync(lead->d_gather + k, lead->device, c->d_partials, c->device, sizeof(fp12), lead->stream));
        CK(cudaMemcpyPeerAsync(lead->d_gather_flags + k, lead->device, c->d_flags, c->device, sizeof(int), lead->stream));
    }
    int bad = 0;
    rc = run_final(lead, (int)ndev, gt_out, &bad, lead->d_gather, lead->d_gather_flags);
    lead->launches = total_launches + lead->launches;
    collect_stage_times(lead, true);
    // the H2D copies of the other devices read the caller's buffer: they are complete (their partials were consumed)
    if (rc < 0) return rc;
    if (bad) { if (gt_out) memset(gt_out, 0, 576); return 0; }
    return rc;
}

extern "C" int blsgpu_batch_verify(blsgpu_ctx *ctx, const void *sets, size_t n, const uint8_t srb[32], uint32_t chunks,
                                   const uint64_t *scalars, uint8_t gt_out[576]) {
    if (!ctx) return BLSGPU_ERR_ARG;
    if (gt_out) memset(gt_out, 0, 576);
    if (n == 0) return 0;
    if (!sets) return fail(ctx, BLSGPU_ERR_ARG, "sets is NULL");
    if (n > blsgpu_capacity(ctx)) return fail(ctx, BLSGPU_ERR_CAPACITY, "batch larger than context capacity");
    // argument errors are reported before the copy is queued: no transfer from the caller's buffer outlives the call
    if (!scalars && !srb) return fail(ctx, BLSGPU_ERR_ARG, "secureRandomBytes is NULL");
    if (scalars)
        for (size_t i = 0; i < n; i++) if (scalars[i] == 0) return fail(ctx, BLSGPU_ERR_ARG, "explicit RLC scalar is zero");
    if (!ctx->peers.empty()) return batch_verify_multi(ctx, (const uint8_t *)sets, n, srb, chunks, scalars, gt_out);
    CK(cudaSetDevice(ctx->device));
    if (batch_plan_of(ctx, n, n, chunks, true, scalars != nullptr).copy_ahead) {
        // small batches replay a captured graph that starts from ctx->d_sets: the copy stays outside of it
        CK(cudaMemcpyAsync(ctx->d_sets, sets, n * sizeof(sigset), cudaMemcpyHostToDevice, ctx->stream));
        return blsgpu_batch_verify_dev(ctx, ctx->d_sets, n, srb, chunks, scalars, gt_out);
    }
    ctx->h_src = (const uint8_t *)sets;                      // run_partial_impl issues the copy (whole, or in overlapped pieces)
    int rc = blsgpu_batch_verify_dev(ctx, ctx->d_sets, n, srb, chunks, scalars, gt_out);
    ctx->h_src = nullptr;
    return rc;
}

extern "C" int blsgpu_partial(blsgpu_ctx *ctx, const void *sets, int sets_on_device, size_t n, size_t first,
                              size_t total_n, const uint8_t srb[32], uint32_t chunks, const uint64_t *scalars,
                              uint8_t partial_out[576], int *flags) {
    if (!ctx || !partial_out) return BLSGPU_ERR_ARG;
    if (n > ctx->cap) return fail(ctx, BLSGPU_ERR_CAPACITY, "share larger than context capacity");
    if (first + n > total_n) return fail(ctx, BLSGPU_ERR_ARG, "share outside the batch");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    if (flags) *flags = 0;
    if (n == 0) {
        // an empty share contributes the neutral element: GT one, in the in-memory (Montgomery) layout
        fp12 one;
        memset(&one, 0, sizeof one);
        CK(cudaMemcpyFromSymbol(&one.c0.c0.c0, FP_ONE, sizeof(fp)));
        memcpy(partial_out, &one, 576);
        return 0;
    }
    const sigset *d = (const sigset *)sets;
    if (sets_on_device && ((uintptr_t)sets & 15)) return fail(ctx, BLSGPU_ERR_ARG, "device sets pointer must be 16-byte aligned (TMA staging)");
    if (!sets_on_device) {
        if (!sets) return fail(ctx, BLSGPU_ERR_ARG, "sets is NULL");
        ctx->h_src = (const uint8_t *)sets;                  // run_partial_impl issues the copy (whole, or in overlapped pieces)
        d = ctx->d_sets;
    }
    int rc = run_partial(ctx, d, n, first, total_n, srb, chunks, scalars, 0);
    ctx->h_src = nullptr;
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->d_partials, 576, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(ctx->h_pinned + 576, ctx->d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    collect_stage_times(ctx, false);
    memcpy(partial_out, ctx->h_pinned, 576);
    int f[4];
    memcpy(f, ctx->h_pinned + 576, sizeof f);
    if (flags) *flags = f[0];
    if (f[0]) memset(partial_out, 0, 576);                  // sealed like blsgpu_partial_dev: zero absorbs the product
    return 0;
}

extern "C" int blsgpu_partial_dev(blsgpu_ctx *ctx, const void *d_sets, size_t n, size_t first, size_t total_n,
                                  const uint8_t srb[32], uint32_t chunks, void *d_partial_out, int *d_flag_out) {
    if (!ctx || !d_partial_out) return BLSGPU_ERR_ARG;
    if (n > ctx->cap) return fail(ctx, BLSGPU_ERR_CAPACITY, "share larger than context capacity");
    if (first + n > total_n) return fail(ctx, BLSGPU_ERR_ARG, "share outside the batch");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    if (n == 0) {
        k_partial_one<<<1, 32, 0, s>>>((fp12 *)d_partial_out, d_flag_out);
        CK(cudaGetLastError());
        ctx->launches = 1;
        return 0;
    }
    if (!d_sets) return fail(ctx, BLSGPU_ERR_ARG, "sets is NULL");
    if ((uintptr_t)d_sets & 15) return fail(ctx, BLSGPU_ERR_ARG, "device sets pointer must be 16-byte aligned (TMA staging)");
    int rc = run_partial(ctx, (const sigset *)d_sets, n, first, total_n, srb, chunks, nullptr, 0);
    if (rc) return rc;
    CK(cudaMemcpyAsync(d_partial_out, ctx->d_partials, 576, cudaMemcpyDeviceToDevice, s));
    k_partial_seal<<<1, 32, 0, s>>>(ctx->d_flags, (uint32_t *)d_partial_out, d_flag_out);
    ctx->launches++;
    CK(cudaGetLastError());
    return 0;
}

extern "C" int blsgpu_finalize_dev(blsgpu_ctx *ctx, const void *d_partials, size_t count, const int *d_flags,
                                   uint8_t gt_out[576]) {
    if (!ctx || !d_partials) return BLSGPU_ERR_ARG;
    if (gt_out) memset(gt_out, 0, 576);
    if (count == 0) return 0;
    if (count > (size_t)INT_MAX) return fail(ctx, BLSGPU_ERR_ARG, "too many partials");
    CK(cudaSetDevice(ctx->device));
    int bad = 0;
    int rc = run_final(ctx, (int)count, gt_out, d_flags ? &bad : nullptr, (const fp12 *)d_partials, d_flags);
    collect_stage_times(ctx, true);
    if (rc < 0) return rc;
    if (bad) { if (gt_out) memset(gt_out, 0, 576); return 0; }
    return rc;
}

extern "C" int blsgpu_finalize(blsgpu_ctx *ctx, const uint8_t *partials, size_t count, uint8_t gt_out[576]) {
    if (!ctx || !partials) return BLSGPU_ERR_ARG;
    if (gt_out) memset(gt_out, 0, 576);
    if (count == 0) return 0;
    if (count > 64) return fail(ctx, BLSGPU_ERR_ARG, "at most 64 partials");
    CK(cudaSetDevice(ctx->device));
    ctx->launches = 0;
    CK(cudaMemcpyAsync(ctx->d_partials, partials, count * 576, cudaMemcpyHostToDevice, ctx->stream));
    int rc = run_final(ctx, (int)count, gt_out, nullptr);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev[2 * ST_FINAL], ctx->ev[2 * ST_FINAL + 1]) == cudaSuccess) ctx->stage_ms[ST_FINAL] = ms;
    return rc;
}

extern "C" int blsgpu_hash_to_g2(blsgpu_ctx *ctx, const uint8_t *msgs, size_t n, size_t msg_len, const uint8_t *dst,
                                 size_t dst_len, uint8_t *out_compressed, uint8_t *out_affine) {
    if (!ctx || (!msgs && msg_len) || !dst) return BLSGPU_ERR_ARG;
    if (dst_len > 255) return fail(ctx, BLSGPU_ERR_ARG, "DST longer than 255 bytes is not supported");
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    size_t o_msgs = 0, o_dst = (n * msg_len + 255) & ~(size_t)255, o_aff = o_dst + 256, o_comp = o_aff + n * 192;
    int rc = ensure_misc(ctx, o_comp + n * 96);
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    if (msg_len) CK(cudaMemcpyAsync(base + o_msgs, msgs, n * msg_len, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(base + o_dst, dst, dst_len, cudaMemcpyHostToDevice, s));
    k_hash_to_g2<<<nblk(n), 128, 0, s>>>(base + o_msgs, n, msg_len, nullptr, base + o_dst, (uint32_t)dst_len,
                                         out_affine ? (g2_aff *)(base + o_aff) : nullptr, out_compressed ? base + o_comp : nullptr);
    CK(cudaGetLastError());
    if (out_affine) CK(cudaMemcpyAsync(out_affine, base + o_aff, n * 192, cudaMemcpyDeviceToHost, s));
    if (out_compressed) CK(cudaMemcpyAsync(out_compressed, base + o_comp, n * 96, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}

// Test hook: the hash of the small-batch route up to (and including) the cofactor-clearing program.
// out_in / out_out: n x 6 field elements each (homogeneous point before / after the program), host buffers.
extern "C" int blsgpu_test_small_hash(blsgpu_ctx *ctx, const void *sets320, size_t n, uint8_t *out_in, uint8_t *out_out) {
    if (!ctx || !sets320 || n == 0 || n > route::SMALL_ROUTE_CAP || n > ctx->cap) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    small_bufs sb;
    int rc = small_buffers(ctx, sb);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->d_sets, sets320, n * 320, cudaMemcpyHostToDevice, s));
    rc = launch_small_hash(ctx, sb, s, n, ctx->d_sets, nullptr, nullptr, nullptr, 0);
    if (rc) return rc;
    CK(cudaGetLastError());
    if (out_in) CK(cudaMemcpyAsync(out_in, sb.hash_in, n * 6 * sizeof(fp), cudaMemcpyDeviceToHost, s));
    if (out_out) CK(cudaMemcpyAsync(out_out, sb.hash_out, n * 6 * sizeof(fp), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int blsgpu_aggregate_g1(blsgpu_ctx *ctx, const void *points96, size_t n, uint8_t out96[96]) {
    if (!ctx || !out96) return BLSGPU_ERR_ARG;
    if (n == 0) return 0;                                   // blst_min_pubkey_sig_core.nim:183-184
    if (!points96) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    int rc = ensure_misc(ctx, n * (sizeof(g1_aff) + sizeof(g1_jac)) + 256);
    if (rc) return rc;
    g1_jac *J = (g1_jac *)ctx->d_misc;
    g1_aff *A = (g1_aff *)((uint8_t *)ctx->d_misc + n * sizeof(g1_jac));
    CK(cudaMemcpyAsync(A, points96, n * sizeof(g1_aff), cudaMemcpyHostToDevice, s));
    k_g1_load<<<nblk(n), 128, 0, s>>>(A, n, J);
    for (size_t m = n; m > 1;) { size_t half = (m + 1) / 2; k_g1_tree<<<nblk(half), 128, 0, s>>>(J, m, half); m = half; }
    k_g1_to_affine<<<1, 32, 0, s>>>(J, A);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out96, A, 96, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 1;
}

extern "C" int blsgpu_aggregate_g2(blsgpu_ctx *ctx, const void *points192, size_t n, uint8_t out192[192]) {
    if (!ctx || !out192) return BLSGPU_ERR_ARG;
    if (n == 0) return 0;
    if (!points192) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    int rc = ensure_misc(ctx, n * (sizeof(g2_aff) + sizeof(g2_jac)) + 256);
    if (rc) return rc;
    g2_jac *J = (g2_jac *)ctx->d_misc;
    g2_aff *A = (g2_aff *)((uint8_t *)ctx->d_misc + n * sizeof(g2_jac));
    CK(cudaMemcpyAsync(A, points192, n * sizeof(g2_aff), cudaMemcpyHostToDevice, s));
    k_g2_load<<<nblk(n), 128, 0, s>>>(A, n, J);
    for (size_t m = n; m > 1;) { size_t half = (m + 1) / 2; k_g2_tree<<<nblk(half), 128, 0, s>>>(J, m, half); m = half; }
    k_g2_to_affine<<<1, 32, 0, s>>>(J, A);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out192, A, 192, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 1;
}

// ---- SURVEY §8f N1: subtractAll (blst_min_pubkey_sig_core.nim:197-209) ----
// dst - sum(elems) computed as -((sum(elems)) + (-dst)): one tree over n + 1 points with the negated dst in the last
// slot, one negation of the root, one inversion.  Affine output, hence bit-identical to the reference's
// aggregate / cneg / aggregate(dst) / finish sequence whatever the order of the additions.
template <class F> static int subtract_all(blsgpu_ctx *ctx, void *dst, const void *elems, size_t n,
                                           void (*load)(const aff_t<F> *, size_t, jac_t<F> *, cudaStream_t),
                                           void (*tree)(jac_t<F> *, size_t, size_t, cudaStream_t),
                                           void (*to_affine)(const jac_t<F> *, aff_t<F> *, cudaStream_t)) {
    if (!ctx || !dst) return BLSGPU_ERR_ARG;
    if (n == 0) return 1;                                   // :199-200: dst untouched
    if (!elems) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    size_t m = n + 1;
    int rc = ensure_misc(ctx, m * (sizeof(aff_t<F>) + sizeof(jac_t<F>)) + 256);
    if (rc) return rc;
    jac_t<F> *J = (jac_t<F> *)ctx->d_misc;
    aff_t<F> *A = (aff_t<F> *)((uint8_t *)ctx->d_misc + m * sizeof(jac_t<F>));
    CK(cudaMemcpyAsync(A, elems, n * sizeof(aff_t<F>), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(A + n, dst, sizeof(aff_t<F>), cudaMemcpyHostToDevice, s));
    load(A, m, J, s);
    k_pt_neg<F><<<1, 32, 0, s>>>(J + n);
    for (size_t k = m; k > 1;) { size_t half = (k + 1) / 2; tree(J, k, half, s); k = half; }
    k_pt_neg<F><<<1, 32, 0, s>>>(J);
    to_affine(J, A, s);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(dst, A, sizeof(aff_t<F>), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 1;
}

extern "C" int blsgpu_subtract_g1(blsgpu_ctx *ctx, uint8_t dst96[96], const void *elems96, size_t n) {
    return subtract_all<fp>(
        ctx, dst96, elems96, n,
        [](const g1_aff *a, size_t m, g1_jac *j, cudaStream_t s) { k_g1_load<<<nblk(m), 128, 0, s>>>(a, m, j); },
        [](g1_jac *j, size_t k, size_t half, cudaStream_t s) { k_g1_tree<<<nblk(half), 128, 0, s>>>(j, k, half); },
        [](const g1_jac *j, g1_aff *a, cudaStream_t s) { k_g1_to_affine<<<1, 32, 0, s>>>(j, a); });
}

extern "C" int blsgpu_subtract_g2(blsgpu_ctx *ctx, uint8_t dst192[192], const void *elems192, size_t n) {
    return subtract_all<fp2>(
        ctx, dst192, elems192, n,
        [](const g2_aff *a, size_t m, g2_jac *j, cudaStream_t s) { k_g2_load<<<nblk(m), 128, 0, s>>>(a, m, j); },
        [](g2_jac *j, size_t k, size_t half, cudaStream_t s) { k_g2_tree<<<nblk(half), 128, 0, s>>>(j, k, half); },
        [](const g2_jac *j, g2_aff *a, cudaStream_t s) { k_g2_to_affine<<<1, 32, 0, s>>>(j, a); });
}

// ---- SURVEY §8f N3: aggregateVerify / fastAggregateVerify on the device ----
// d_pks: n affine public keys on the device; messages/DST/signature are staged into d_misc by the callers below.
static int verify_pairs_dev(blsgpu_ctx *ctx, const g1_aff *d_pks, size_t n, const uint8_t *d_msgs, const uint32_t *d_offs,
                            const uint8_t *d_dst, size_t dst_len, const g2_aff *d_sig, uint8_t gt_out[576]) {
    cudaStream_t s = ctx->stream;
    ctx->launches = 0;
    CK(cudaMemsetAsync(ctx->d_flags, 0, 4 * sizeof(int), s));
    BEGIN(ST_HASH, s);
    if (route::program_hash(thr(), n, ctx->serial_tail)) {
        small_bufs sb;
        int rcp = small_buffers(ctx, sb);
        if (!rcp) rcp = launch_small_hash(ctx, sb, s, n, nullptr, d_msgs, d_offs, d_dst, dst_len);
        if (rcp) return rcp;
        k_g2_hom_to_affine<<<(unsigned)n, 32, 0, s>>>(sb.hash_out, n, ctx->d_Q);
        ctx->launches += 2;                                 // the map and the conversion
    } else {
        k_hash_to_g2<<<nblk(n), 128, 0, s>>>(d_msgs, n, 0, d_offs, d_dst, (uint32_t)dst_len, ctx->d_Q, nullptr);
    }
    END(ST_HASH, s);
    k_verify_pairs<<<nblk(n + 1), 128, 0, s>>>(d_pks, n, d_sig, ctx->d_Q, ctx->d_P, ctx->d_flags);
    ctx->launches += 2;
    CK(cudaGetLastError());
    int rc = run_miller(ctx, ctx->ml, n + 1, 0);
    if (rc) return rc;
    int pk_inf = 0;
    rc = run_final(ctx, 1, gt_out, &pk_inf);
    if (rc < 0) return rc;
    if (pk_inf) { if (gt_out) memset(gt_out, 0, 576); return 0; }
    return rc;
}

// host staging layout in d_misc: [msgs | offsets | dst | sig | pks]; returns device pointers
struct verify_stage { uint8_t *msgs; uint32_t *offs; uint8_t *dst; g2_aff *sig; g1_aff *pks; };
static int stage_verify_inputs(blsgpu_ctx *ctx, const void *pks, size_t npk, const uint8_t *msgs, size_t msg_bytes,
                               const uint32_t *offs, size_t noffs, const uint8_t *dst, size_t dst_len, const void *sig,
                               size_t extra, verify_stage &st, uint8_t **extra_ptr) {
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t o_msgs = 0, o_offs = up(msg_bytes + 1), o_dst = o_offs + up(noffs * 4), o_sig = o_dst + up(dst_len + 1),
           o_pks = o_sig + 256, o_extra = o_pks + up(npk * 96), total = o_extra + up(extra);
    int rc = ensure_misc(ctx, total);
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    cudaStream_t s = ctx->stream;
    st.msgs = base + o_msgs; st.offs = (uint32_t *)(base + o_offs); st.dst = base + o_dst;
    st.sig = (g2_aff *)(base + o_sig); st.pks = (g1_aff *)(base + o_pks);
    if (extra_ptr) *extra_ptr = base + o_extra;
    if (msg_bytes) CK(cudaMemcpyAsync(st.msgs, msgs, msg_bytes, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(st.offs, offs, noffs * 4, cudaMemcpyHostToDevice, s));
    if (dst_len) CK(cudaMemcpyAsync(st.dst, dst, dst_len, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(st.sig, sig, 192, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(st.pks, pks, npk * 96, cudaMemcpyHostToDevice, s));
    return 0;
}

extern "C" int blsgpu_aggregate_verify(blsgpu_ctx *ctx, const void *pubkeys96, size_t n, const uint8_t *msgs,
                                       const uint32_t *msg_offsets, const uint8_t *dst, size_t dst_len, const void *sig192,
                                       uint8_t gt_out[576]) {
    if (!ctx) return BLSGPU_ERR_ARG;
    if (gt_out) memset(gt_out, 0, 576);
    if (n == 0) return 0;                                   // bls_sig_min_pubkey.nim:140, :167, :189
    if (!pubkeys96 || !msg_offsets || !sig192 || (!dst && dst_len)) return fail(ctx, BLSGPU_ERR_ARG, "NULL argument");
    if (dst_len > 255) return fail(ctx, BLSGPU_ERR_ARG, "DST longer than 255 bytes is not supported");
    if (n > ctx->cap) return fail(ctx, BLSGPU_ERR_CAPACITY, "more pairs than the context capacity");
    for (size_t i = 0; i < n; i++)
        if (msg_offsets[i + 1] < msg_offsets[i]) return fail(ctx, BLSGPU_ERR_ARG, "message offsets must be non-decreasing");
    if (msg_offsets[n] && !msgs) return fail(ctx, BLSGPU_ERR_ARG, "msgs is NULL");
    CK(cudaSetDevice(ctx->device));
    verify_stage st;
    int rc = stage_verify_inputs(ctx, pubkeys96, n, msgs, msg_offsets[n], msg_offsets, n + 1, dst, dst_len, sig192, 0, st, nullptr);
    if (rc) return rc;
    rc = verify_pairs_dev(ctx, st.pks, n, st.msgs, st.offs, st.dst, dst_len, st.sig, gt_out);
    collect_stage_times(ctx, true);
    return rc;
}

extern "C" int blsgpu_fast_aggregate_verify(blsgpu_ctx *ctx, const void *pubkeys96, size_t n, const uint8_t *msg,
                                            size_t msg_len, const uint8_t *dst, size_t dst_len, const void *sig192,
                                            uint8_t gt_out[576]) {
    if (!ctx) return BLSGPU_ERR_ARG;
    if (gt_out) memset(gt_out, 0, 576);
    if (n == 0) return 0;                                   // bls_sig_min_pubkey.nim:251-253
    if (!pubkeys96 || !sig192 || (!msg && msg_len) || (!dst && dst_len)) return fail(ctx, BLSGPU_ERR_ARG, "NULL argument");
    if (dst_len > 255) return fail(ctx, BLSGPU_ERR_ARG, "DST longer than 255 bytes is not supported");
    if (msg_len > 0xffffffffu || n > 0xffffffffu) return fail(ctx, BLSGPU_ERR_ARG, "input too large");
    CK(cudaSetDevice(ctx->device));
    const uint32_t offs[4] = {0, (uint32_t)msg_len, 0, (uint32_t)n};       // message offsets | key-segment offsets
    verify_stage st;
    uint8_t *extra = nullptr;
    int rc = stage_verify_inputs(ctx, pubkeys96, n, msg, msg_len, offs, 4, dst, dst_len, sig192, 512, st, &extra);
    if (rc) return rc;
    cudaStream_t s = ctx->stream;
    g1_jac *aggj = (g1_jac *)extra;
    g1_aff *agg = (g1_aff *)(extra + 256);
    k_g1_seg_sum<<<1, 128, 0, s>>>(st.pks, st.offs + 2, 1, aggj);      // aggregateAll (blst_min_pubkey_sig_core.nim:179)
    k_g1_to_affine_many<<<1, 128, 0, s>>>(aggj, 1, agg);
    CK(cudaGetLastError());
    rc = verify_pairs_dev(ctx, agg, 1, st.msgs, st.offs, st.dst, dst_len, st.sig, gt_out);
    ctx->launches += 2;
    collect_stage_times(ctx, true);
    return rc;
}

extern "C" int blsgpu_aggregate_g1_segments(blsgpu_ctx *ctx, const void *points96, const uint32_t *offsets, size_t nseg,
                                            uint8_t *out96) {
    if (!ctx || !offsets || !out96) return BLSGPU_ERR_ARG;
    if (nseg == 0) return 0;
    for (size_t i = 0; i < nseg; i++)
        if (offsets[i + 1] < offsets[i]) return fail(ctx, BLSGPU_ERR_ARG, "segment offsets must be non-decreasing");
    const size_t n = offsets[nseg];
    if (n && !points96) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t o_pts = 0, o_offs = up(n * 96 + 1), o_j = o_offs + up((nseg + 1) * 4), o_a = o_j + up(nseg * sizeof(g1_jac));
    int rc = ensure_misc(ctx, o_a + up(nseg * 96));
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    if (n) CK(cudaMemcpyAsync(base + o_pts, points96, n * 96, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(base + o_offs, offsets, (nseg + 1) * 4, cudaMemcpyHostToDevice, s));
    k_g1_seg_sum<<<nblk(nseg, 4), 128, 0, s>>>((const g1_aff *)(base + o_pts), (const uint32_t *)(base + o_offs), nseg,
                                               (g1_jac *)(base + o_j));
    k_g1_to_affine_many<<<nblk(nseg), 128, 0, s>>>((const g1_jac *)(base + o_j), nseg, (g1_aff *)(base + o_a));
    ctx->launches = 2;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out96, base + o_a, nseg * 96, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 1;
}

// ---- SURVEY §8f N2: batched fromBytes with checks ----
template <int G2>
static int from_bytes_api(blsgpu_ctx *ctx, const uint8_t *in, size_t n, size_t in_len, int group_check, uint8_t *out,
                          uint8_t *status) {
    const size_t pb = G2 ? 192 : 96, clen = G2 ? 96 : 48;
    if (!ctx || !out) return BLSGPU_ERR_ARG;
    if (n == 0) return 1;
    if (!in) return BLSGPU_ERR_ARG;
    if (in_len != clen && in_len != pb) return fail(ctx, BLSGPU_ERR_ARG, "encoded length must be the compressed or the serialized size");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    size_t o_in = 0, o_out = up(n * in_len), o_st = o_out + up(n * pb), o_cnt = o_st + up(n);
    int rc = ensure_misc(ctx, o_cnt + 256);
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    CK(cudaMemcpyAsync(base + o_in, in, n * in_len, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(base + o_cnt, 0, 4, s));
    if (G2) k_signatures_from_bytes<<<nblk(n), 128, 0, s>>>(base + o_in, n, (int)in_len, group_check, (g2_aff *)(base + o_out),
                                                            base + o_st, (int *)(base + o_cnt));
    else k_pubkeys_from_bytes<<<nblk(n), 128, 0, s>>>(base + o_in, n, (int)in_len, group_check, (g1_aff *)(base + o_out),
                                                      base + o_st, (int *)(base + o_cnt));
    ctx->launches = 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, base + o_out, n * pb, cudaMemcpyDeviceToHost, s));
    if (status) CK(cudaMemcpyAsync(status, base + o_st, n, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(ctx->h_pinned, base + o_cnt, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    int nfail;
    memcpy(&nfail, ctx->h_pinned, 4);
    return nfail == 0 ? 1 : 0;
}

extern "C" int blsgpu_pubkeys_from_bytes(blsgpu_ctx *ctx, const uint8_t *in, size_t n, size_t in_len, int group_check,
                                         uint8_t *out96, uint8_t *status) {
    return from_bytes_api<0>(ctx, in, n, in_len, group_check, out96, status);
}
extern "C" int blsgpu_signatures_from_bytes(blsgpu_ctx *ctx, const uint8_t *in, size_t n, size_t in_len, int group_check,
                                            uint8_t *out192, uint8_t *status) {
    return from_bytes_api<1>(ctx, in, n, in_len, group_check, out192, status);
}

template <int G2>
static int compress_api(blsgpu_ctx *ctx, const void *points, size_t n, uint8_t *out) {
    const size_t pb = G2 ? 192 : 96, clen = G2 ? 96 : 48;
    if (!ctx || !out) return BLSGPU_ERR_ARG;
    if (n == 0) return 1;
    if (!points) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    size_t o_out = (n * pb + 255) & ~(size_t)255;
    int rc = ensure_misc(ctx, o_out + n * clen + 256);
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    CK(cudaMemcpyAsync(base, points, n * pb, cudaMemcpyHostToDevice, s));
    if (G2) k_g2_compress<<<nblk(n), 128, 0, s>>>((const g2_aff *)base, n, base + o_out);
    else k_g1_compress<<<nblk(n), 128, 0, s>>>((const g1_aff *)base, n, base + o_out);
    ctx->launches = 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, base + o_out, n * clen, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 1;
}
extern "C" int blsgpu_pubkeys_to_bytes(blsgpu_ctx *ctx, const void *points96, size_t n, uint8_t *out48) {
    return compress_api<0>(ctx, points96, n, out48);
}
extern "C" int blsgpu_signatures_to_bytes(blsgpu_ctx *ctx, const void *points192, size_t n, uint8_t *out96) {
    return compress_api<1>(ctx, points192, n, out96);
}

template <class F>
static int msm_api_dev(blsgpu_ctx *ctx, const void *d_points, const void *d_scalars, size_t n, size_t nbits, uint8_t *out) {
    const size_t pb = sizeof(aff_t<F>);
    if (!ctx || !out) return BLSGPU_ERR_ARG;
    memset(out, 0, pb);
    if (n == 0) return 0;
    if (!d_points || !d_scalars || nbits == 0 || nbits > 256) return fail(ctx, BLSGPU_ERR_ARG, "bad MSM arguments");
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_misc2(ctx, 256);
    if (rc) return rc;
    ctx->launches = 0;
    rc = run_msm<F>(ctx, (const uint8_t *)d_points, pb, (const uint8_t *)d_scalars, (nbits + 7) / 8, n, (int)nbits, ctx->stream,
                    nullptr, (aff_t<F> *)ctx->d_misc2);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_pinned, ctx->d_misc2, pb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memcpy(out, ctx->h_pinned, pb);
    return 1;
}

template <class F>
static int msm_api_multi(blsgpu_ctx *lead, const uint8_t *points, const uint8_t *scalars, size_t n, size_t nbits, uint8_t *out);

template <class F>
static int msm_api_host(blsgpu_ctx *ctx, const void *points, const void *scalars, size_t n, size_t nbits, uint8_t *out) {
    const size_t pb = sizeof(aff_t<F>);
    if (!ctx || !out) return BLSGPU_ERR_ARG;
    memset(out, 0, pb);
    if (n == 0) return 0;
    if (!points || !scalars || nbits == 0 || nbits > 256) return fail(ctx, BLSGPU_ERR_ARG, "bad MSM arguments");
    if (!ctx->peers.empty() && n >= 2 * (1 + ctx->peers.size()))
        return msm_api_multi<F>(ctx, (const uint8_t *)points, (const uint8_t *)scalars, n, nbits, out);
    CK(cudaSetDevice(ctx->device));
    size_t sb = (nbits + 7) / 8;
    int rc = ensure_misc(ctx, n * pb + n * sb + 256);
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    CK(cudaMemcpyAsync(base, points, n * pb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(base + n * pb, scalars, n * sb, cudaMemcpyHostToDevice, ctx->stream));
    return msm_api_dev<F>(ctx, base, base + n * pb, n, nbits, out);
}

// MSM over every device of a multi-device context (SURVEY.md section 8e, MSM row): device k takes the k-th balanced
// slice of the points and scalars and returns ONE affine point (unique coordinates: an empty or cancelling share is the
// all-zero point); the leader sums the ndev points with the aggregateAll tree.  All devices are launched before any is
// waited for.
template <class F>
static int msm_api_multi(blsgpu_ctx *lead, const uint8_t *points, const uint8_t *scalars, size_t n, size_t nbits, uint8_t *out) {
    const size_t pb = sizeof(aff_t<F>), sb = (nbits + 7) / 8;
    std::vector<blsgpu_ctx *> all;
    all.push_back(lead);
    for (blsgpu_ctx *p : lead->peers) all.push_back(p);
    const size_t ndev = all.size();
    std::vector<uint8_t> parts(ndev * pb, 0);
    std::vector<char> busy(ndev, 0);
    int rc = 0, launches = 0;
    for (size_t k = 0; k < ndev && rc == 0; k++) {
        blsgpu_ctx *ctx = all[k];
        size_t first, len;
        share_range(n, ndev, k, first, len);
        if (len == 0) continue;
        cudaError_t e = cudaSetDevice(ctx->device);
        if (e != cudaSuccess) { rc = fail(lead, BLSGPU_ERR_CUDA, "cudaSetDevice", e); break; }
        rc = ensure_misc(ctx, len * pb + len * sb + 256);
        if (!rc) rc = ensure_misc2(ctx, 256);
        if (rc) break;
        uint8_t *base = (uint8_t *)ctx->d_misc;
        if ((e = cudaMemcpyAsync(base, points + first * pb, len * pb, cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess ||
            (e = cudaMemcpyAsync(base + len * pb, scalars + first * sb, len * sb, cudaMemcpyHostToDevice, ctx->stream)) != cudaSuccess) {
            rc = fail(lead, BLSGPU_ERR_CUDA, "cudaMemcpyAsync(msm share)", e);
            break;
        }
        busy[k] = 1;
        ctx->launches = 0;
        int r = run_msm<F>(ctx, base, pb, base + len * pb, sb, len, (int)nbits, ctx->stream, nullptr, (aff_t<F> *)ctx->d_misc2);
        if (r) { rc = fail(lead, r, ctx->err.c_str()); break; }
        launches += ctx->launches;
        if ((e = cudaMemcpyAsync(ctx->h_pinned, ctx->d_misc2, pb, cudaMemcpyDeviceToHost, ctx->stream)) != cudaSuccess)
            rc = fail(lead, BLSGPU_ERR_CUDA, "cudaMemcpyAsync(msm partial)", e);
    }
    for (size_t k = 0; k < ndev; k++) {
        if (!busy[k]) continue;
        cudaSetDevice(all[k]->device);
        cudaError_t e = cudaStreamSynchronize(all[k]->stream);
        if (e != cudaSuccess && rc == 0) rc = fail(lead, BLSGPU_ERR_CUDA, "cudaStreamSynchronize(msm share)", e);
        if (rc == 0) memcpy(parts.data() + k * pb, all[k]->h_pinned, pb);
    }
    cudaSetDevice(lead->device);
    if (rc) return rc;
    rc = sizeof(F) == sizeof(fp) ? blsgpu_aggregate_g1(lead, parts.data(), ndev, out) : blsgpu_aggregate_g2(lead, parts.data(), ndev, out);
    lead->launches = launches;
    return rc;
}

extern "C" int blsgpu_msm_g1_dev(blsgpu_ctx *ctx, const void *d_points96, const void *d_scalars, size_t n, size_t nbits,
                                 uint8_t out96[96]) {
    return msm_api_dev<fp>(ctx, d_points96, d_scalars, n, nbits, out96);
}
extern "C" int blsgpu_msm_g1(blsgpu_ctx *ctx, const void *points96, const void *scalars, size_t n, size_t nbits,
                             uint8_t out96[96]) {
    return msm_api_host<fp>(ctx, points96, scalars, n, nbits, out96);
}
extern "C" int blsgpu_msm_g2_dev(blsgpu_ctx *ctx, const void *d_points192, const void *d_scalars, size_t n, size_t nbits,
                                 uint8_t out192[192]) {
    return msm_api_dev<fp2>(ctx, d_points192, d_scalars, n, nbits, out192);
}
extern "C" int blsgpu_msm_g2(blsgpu_ctx *ctx, const void *points192, const void *scalars, size_t n, size_t nbits,
                             uint8_t out192[192]) {
    return msm_api_host<fp2>(ctx, points192, scalars, n, nbits, out192);
}

extern "C" int blsgpu_combine(blsgpu_ctx *ctx, const uint8_t srb[32], const void *pubkeys96, const void *sigs192, size_t n,
                              uint8_t pk_out[96], uint8_t sig_out[192]) {
    if (!ctx || !srb || !pubkeys96 || !sigs192 || !pk_out || !sig_out) return BLSGPU_ERR_ARG;
    if (n == 0) return fail(ctx, BLSGPU_ERR_ARG, "combine: must provide at least 1 signature");   // raiseAssert in the reference
    if (n == 1) { memcpy(pk_out, pubkeys96, 96); memcpy(sig_out, sigs192, 192); return 1; }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    int rc = ensure_misc(ctx, n * (96 + 192 + 8) + 1024);
    if (rc) return rc;
    rc = ensure_misc2(ctx, 1024);
    if (rc) return rc;
    uint8_t *base = (uint8_t *)ctx->d_misc;
    uint8_t *d_sig = base, *d_pk = base + n * 192, *d_sc = base + n * (192 + 96);   // 16-byte aligned blocks
    d_sc = (uint8_t *)(((uintptr_t)d_sc + 15) & ~(uintptr_t)15);
    CK(cudaMemcpyAsync(d_pk, pubkeys96, n * 96, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_sig, sigs192, n * 192, cudaMemcpyHostToDevice, s));
    ctx->launches = 1;
    k_combine_scalars<<<1, 32, 0, s>>>(words_of(srb), n, (uint64_t *)d_sc);
    g1_aff *o1 = (g1_aff *)ctx->d_misc2;
    g2_aff *o2 = (g2_aff *)((uint8_t *)ctx->d_misc2 + 256);
    rc = run_msm<fp>(ctx, d_pk, 96, d_sc, 8, n, 64, s, nullptr, o1);
    if (!rc) rc = run_msm<fp2>(ctx, d_sig, 192, d_sc, 8, n, 64, s, nullptr, o2);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_pinned, o1, 96, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(ctx->h_pinned + 256, o2, 192, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memcpy(pk_out, ctx->h_pinned, 96);
    memcpy(sig_out, ctx->h_pinned + 256, 192);
    return 1;
}

extern "C" int blsgpu_msm_make_inputs(blsgpu_ctx *ctx, uint64_t seed, size_t n, void *d_points96, void *d_scalars32) {
    if (!ctx || !d_points96 || !d_scalars32) return BLSGPU_ERR_ARG;
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    k_msm_make_inputs<<<nblk(n), 128, 0, ctx->stream>>>(seed, n, (g1_aff *)d_points96, (uint8_t *)d_scalars32);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int blsgpu_last_stage_ms(const blsgpu_ctx *ctx, float *ms, int max) {
    if (!ctx || !ms) return 0;
    int k = max < ST_COUNT ? max : ST_COUNT;
    for (int i = 0; i < k; i++) ms[i] = ctx->stage_ms[i];
    return k;
}
extern "C" const char *blsgpu_stage_name(int stage) { return stage >= 0 && stage < ST_COUNT ? STAGE_NAMES[stage] : ""; }
extern "C" int blsgpu_last_launches(const blsgpu_ctx *ctx) { return ctx ? ctx->launches : 0; }

// n records of field test op `op` from d_in to d_out (device scratch), on the context's stream
static int launch_test_field(blsgpu_ctx *ctx, int op, const uint8_t *d_in, size_t n, uint8_t *d_out) {
    const test_field_shape &sh = TEST_FIELD_OPS[op];
    const size_t per_block = sh.geom == TF_THREAD ? ACC_BS : sh.geom == TF_PAIR ? ACC_BS / 2
                           : sh.geom == TF_TEAM_LANE ? 6 * ACC_TPB : ACC_TPB;
    k_test_field<<<nblk(n, (unsigned)per_block), ACC_BS, 0, ctx->stream>>>(op, d_in, test_field_rec(sh.nin, sh.nin_w), n, d_out,
                                                                         test_field_rec(sh.nout, sh.nout_w));
    CK(cudaGetLastError());
    return 0;
}

extern "C" int blsgpu_test_field(blsgpu_ctx *ctx, int op, const void *in, size_t in_rec_bytes, size_t n, void *out,
                                 size_t out_rec_bytes) {
    if (!ctx) return BLSGPU_ERR_ARG;
    if (op < 0 || op >= BLSGPU_TF_COUNT) return fail(ctx, BLSGPU_ERR_ARG, "unknown field test op");
    const test_field_shape &sh = TEST_FIELD_OPS[op];
    if (in_rec_bytes != test_field_rec(sh.nin, sh.nin_w) || out_rec_bytes != test_field_rec(sh.nout, sh.nout_w))
        return fail(ctx, BLSGPU_ERR_ARG, "record size does not match the field test op");
    if (n == 0) return 0;
    if (!in || !out) return BLSGPU_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    int rc = ensure_misc(ctx, n * (in_rec_bytes + out_rec_bytes));
    if (rc) return rc;
    uint8_t *d_in = (uint8_t *)ctx->d_misc, *d_out = d_in + n * in_rec_bytes;
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpyAsync(d_in, in, n * in_rec_bytes, cudaMemcpyHostToDevice, s));
    rc = launch_test_field(ctx, op, d_in, n, d_out);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_out, n * out_rec_bytes, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int blsgpu_test_fp(blsgpu_ctx *ctx, int op, const void *a, const void *b, size_t n, void *out) {
    if (!ctx || !a || !out) return BLSGPU_ERR_ARG;
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    const int fop = op == 0 ? BLSGPU_TF_FP_MUL : op == 1 ? BLSGPU_TF_FP_ADD : op == 2 ? BLSGPU_TF_FP_SUB
                  : op == 3 ? BLSGPU_TF_FP_SQR : op == 6 ? BLSGPU_TF_FP_INV_VARTIME : BLSGPU_TF_FP_INV;
    const size_t rec = 48 * (size_t)TEST_FIELD_OPS[fop].nin;   // a, or a and b (b = a when NULL) side by side
    int rc = ensure_misc(ctx, n * (rec + 48));
    if (rc) return rc;
    uint8_t *d_in = (uint8_t *)ctx->d_misc, *d_out = d_in + n * rec;
    cudaStream_t s = ctx->stream;
    CK(cudaMemcpy2DAsync(d_in, rec, a, 48, 48, n, cudaMemcpyHostToDevice, s));
    if (rec == 96) CK(cudaMemcpy2DAsync(d_in + 48, rec, b ? b : a, 48, 48, n, cudaMemcpyHostToDevice, s));
    rc = launch_test_field(ctx, fop, d_in, n, d_out);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out, d_out, n * 48, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}

extern "C" double blsgpu_imad_peak(blsgpu_ctx *ctx, int wide) {
    if (!ctx) return -1.0;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return -1.0;
    if (ensure_misc(ctx, 256)) return -1.0;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ctx->device) != cudaSuccess) return -1.0;
    const int iters = 4096, blocks = prop.multiProcessorCount * 8, threads = 256;
    cudaStream_t s = ctx->stream;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(e0, s);
        if (wide) k_imad_peak<1><<<blocks, threads, 0, s>>>((uint32_t *)ctx->d_misc, iters, 12345u + rep);
        else k_imad_peak<0><<<blocks, threads, 0, s>>>((uint32_t *)ctx->d_misc, iters, 12345u + rep);
        cudaEventRecord(e1, s);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double ops = (double)blocks * threads * iters * 64.0;
        double rate = ops / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return best;
}

extern "C" double blsgpu_fpmul_peak(blsgpu_ctx *ctx, int threads_per_block, int blocks_per_sm) {
    if (!ctx) return -1.0;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return -1.0;
    if (ensure_misc(ctx, 256)) return -1.0;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ctx->device) != cudaSuccess) return -1.0;
    const int iters = 2000, blocks = prop.multiProcessorCount * blocks_per_sm;
    cudaStream_t s = ctx->stream;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 4; rep++) {
        cudaEventRecord(e0, s);
        k_fpmul_peak<<<blocks, threads_per_block, 0, s>>>((fp *)ctx->d_misc, iters, 99u + rep);
        cudaEventRecord(e1, s);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double rate = (double)blocks * threads_per_block * iters * 2.0 / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return best;
}

extern "C" int blsgpu_make_sets(blsgpu_ctx *ctx, uint64_t seed, size_t first, size_t n, void *out, int out_on_device) {
    if (!ctx || !out) return BLSGPU_ERR_ARG;
    if (n == 0) return 0;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    sigset *d = (sigset *)out;
    if (!out_on_device) {
        if (n > ctx->cap) return fail(ctx, BLSGPU_ERR_CAPACITY, "batch larger than context capacity");
        d = ctx->d_sets;
    }
    uint8_t sb[32] = {0};
    memcpy(sb, &seed, 8);
    k_make_sets<<<nblk(n), 128, 0, s>>>(words_of(sb), first, n, d);
    CK(cudaGetLastError());
    if (!out_on_device) CK(cudaMemcpyAsync(out, d, n * sizeof(sigset), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}
