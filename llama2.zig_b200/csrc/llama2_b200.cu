// llama2_b200.cu — C ABI (include/llama2_b200.h) over the sm_100a kernels in l2b_device.cuh.
//
// Replaces transformer() of the reference (src/main.zig:285-430) and the device-side
// equivalents of Weights.init (:73-115) / RunState.init (:137-154).  Pure CUDA runtime:
// no torch, no CPU fallback.  One rank = one GPU = one stream; a decode step is a CUDA graph
// of 5 kernels per layer + classifier, replayed per token.  A context is either one rank
// (single GPU, or one process per GPU with peers reached through CUDA IPC) or a group of ranks
// inside one process (l2b_create with n_gpus > 1: peers reached through UVA peer access).
#include "../../include/llama2_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <memory>
#include <set>
#include <string>
#include <vector>

#include "l2b_device.cuh"
#include "l2b_prefill.cuh"

using namespace l2b;

// ---------------------------------------------------------------------------------------
// NCCL through dlopen: single-GPU use never needs libnccl (or its headers) to be present.  NCCL
// is only the bootstrap of the one-process-per-GPU mode (it carries the CUDA IPC handles at
// create time) and the data plane of the L2B_TP=nccl baseline; the default data plane is this
// library's own peer-memory exchange.  The few types / enum values used are restated here.
// ---------------------------------------------------------------------------------------
namespace {
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
constexpr int ncclSuccess = 0;
constexpr int ncclChar = 0, ncclInt = 2, ncclUint64 = 5, ncclFloat = 7;   // ncclDataType_t
constexpr int ncclSum = 0, ncclMax = 2;                                   // ncclRedOp_t

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi g_nccl;

bool nccl_load(std::string *err) {
    if (g_nccl.ok) return true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
        g_nccl.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.handle) break;
    }
    if (!g_nccl.handle) {
        if (err) *err = std::string("dlopen(libnccl.so.2) failed: ") + dlerror();
        return false;
    }
#define L2B_SYM(field, name)                                                        \
    *(void **)(&g_nccl.field) = dlsym(g_nccl.handle, name);                         \
    if (!g_nccl.field) {                                                            \
        if (err) *err = std::string("dlsym failed: ") + name;                       \
        return false;                                                               \
    }
    L2B_SYM(GetUniqueId, "ncclGetUniqueId");
    L2B_SYM(CommInitRank, "ncclCommInitRank");
    L2B_SYM(CommDestroy, "ncclCommDestroy");
    L2B_SYM(AllReduce, "ncclAllReduce");
    L2B_SYM(AllGather, "ncclAllGather");
    L2B_SYM(GetErrorString, "ncclGetErrorString");
#undef L2B_SYM
    g_nccl.ok = true;
    return true;
}
}  // namespace

// ---------------------------------------------------------------------------------------
// Context (one rank)
// ---------------------------------------------------------------------------------------
enum StepMode { MODE_LOGITS = 0, MODE_ARGMAX = 1, MODE_SAMPLE = 2, MODE_NOCLS = 3 };
enum GraphId { G_LOGITS = 0, G_ARGMAX_ONE = 1, G_ARGMAX_LOOP = 2, G_SAMPLE = 3, G_PREFILL_LOOP = 4, G_COUNT = 5 };
constexpr int kCandCap = 8192;               // top-p candidates returned per step (more => host filters itself)

// Device weights (Weights, src/main.zig:53-71) of one single-GPU context, shared by every decode stream
// created over them (l2b_create_stream) and freed with the last context that uses them.  The scratch
// of batched passes (prefill chunks, batched decode steps) lives here too: contexts over one set of
// weights are driven from one thread and every call synchronises before it returns.
struct WeightStore {
    int device = 0;
    std::vector<void *> owned;               // weight tensors and batch scratch (device)
    std::vector<void *> pinned;              // batch scratch (pinned host)
    bool batch_ready = false;
    // [L2B_MAX_BATCH] vectors of dim | q | q | hidden | vocab floats
    float *x = nullptr, *q = nullptr, *xb = nullptr, *hb = nullptr, *logits = nullptr;
    float *part_o = nullptr, *part_ml = nullptr; // attention partials per vector
    unsigned int *counters = nullptr;
    unsigned long long *amax = nullptr;      // [L2B_MAX_BATCH] packed argmax keys
    BatchVec *vec = nullptr;                 // [max(seq_len, L2B_MAX_BATCH)] per-vector table
    int *forced = nullptr, *out = nullptr;   // [L2B_MAX_BATCH][seq_len]
    int *n_done = nullptr;                   // [L2B_MAX_BATCH]
    BatchVec *h_vec = nullptr;               // pinned mirrors
    float *h_logits = nullptr;               // [L2B_MAX_BATCH][vocab]
    int *h_ints = nullptr;                   // [L2B_MAX_BATCH][seq_len] tokens, then [L2B_MAX_BATCH] step counts
    ~WeightStore() {
        cudaSetDevice(device);
        for (void *p : owned) cudaFree(p);
        for (void *p : pinned) cudaFreeHost(p);
    }
};

struct l2b_ctx {
    l2b_config cfg{};
    int rank = 0, world = 1, device = 0, num_sms = 0;
    // in-process group (l2b_create with n_gpus > 1): the leader (rank 0) owns the other ranks
    std::vector<l2b_ctx *> members;          // leader only: all ranks, [0] == this
    l2b_ctx *leader = nullptr;
    // derived sizes (local = this rank's shard)
    int dim = 0, hidden = 0, head_size = 0, kv_mul = 0;
    int q_dim = 0, kv_dim = 0;              // global
    int q_loc = 0, kv_loc = 0, hid_loc = 0, heads_loc = 0, vocab_loc = 0;
    // device weights (Weights, src/main.zig:53-71), this rank's slices, owned by `weights`
    std::shared_ptr<WeightStore> weights;
    float *emb = nullptr, *rms_att = nullptr, *rms_ffn = nullptr, *rms_final = nullptr;
    float *wq = nullptr, *wk = nullptr, *wv = nullptr, *wo = nullptr;
    float *w1 = nullptr, *w2 = nullptr, *w3 = nullptr, *wcls = nullptr;
    // device run state (RunState, :119-135)
    float *X = nullptr;                      // residual stream x; wo / w2 add into it (:395, :422)
    float *Xalt = nullptr;                   // second copy: kernels that fold partial vectors in write the new x here (ping-pong)
    float *final_X = nullptr;                // which of the two holds x after a step
    float *attn_parts = nullptr;             // small-model fusion: (n_heads, dim) partial vectors of attention + wo
    bool fuse_attn = false;
    // batched passes (l2b_prefill, l2b_forward_batch, l2b_generate_argmax_batch) on bandwidth-bound
    // shapes: PF_MAXB vectors per pass over the weights, scratch in `weights`
    bool pf_ready = false, pf_ok = false;
    int attn_R = 1;                          // CTAs per head cluster of attn_wo_kernel
    float *delta = nullptr;                  // L2B_TP=nccl baseline only: partial rows before the NCCL all-reduce
    float *q = nullptr, *xb = nullptr, *hb = nullptr, *logits = nullptr, *logits_loc = nullptr;
    float *kcache = nullptr, *vcache = nullptr;     // (L, seq_len, kv_loc)
    float *rope_cos = nullptr, *rope_sin = nullptr; // (seq_len, head_size/2)
    float *part_o = nullptr, *part_ml = nullptr;
    unsigned int *counters = nullptr;
    int *ctl = nullptr;
    unsigned long long *amax = nullptr;
    int *gen_forced = nullptr, *gen_out = nullptr, *gen_ndone = nullptr;
    ProbIndex *cand = nullptr;               // sampler: top-p candidates (index order)
    int *n_cand = nullptr;
    // host pinned
    float *h_logits = nullptr;               // vocab floats: logits, or probabilities after sample_prep
    int *h_ctl = nullptr;                    // [0..7] host -> device control words, [8..15] device -> host status
    int *h_ints = nullptr;                   // [0]=next, [1]=n_done, [2]=n_cand
    int *h_gen = nullptr;                    // seq_len ints
    ProbIndex *h_cand = nullptr;
    // attention launch shape
    int nsplit = 1, min_chunk = 256, attn_smem = 0;   // timeline splits of >= 256 positions
    // streams / graphs
    cudaStream_t stream = nullptr;
    cudaGraphExec_t graphs[G_COUNT] = {};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool use_graphs = true;
    bool use_pdl = true;
    bool time_steps = false;                 // L2B_TIME_STEPS=1: CUDA events around every single step (l2b_last_timing)
    int last_grid = 0;                       // grid of the most recent GEMV launch
    // tensor-parallel exchange over peer memory (world > 1).  One arena per rank holds every landing
    // area, so one IPC handle (or one UVA pointer) per rank is all the ranks trade at create time:
    //   ll_red    [2L reduce points][world source ranks][dim] LL units   (wo / w2 partial rows)
    //   ll_logits [vocab] LL units                                       (classifier slices of all ranks)
    //   ll_amax   [world][2] LL units                                    (packed argmax keys)
    bool use_p2p = false;
    unsigned char *arena = nullptr;
    size_t arena_bytes = 0, off_red = 0, off_logits = 0, off_amax = 0;
    unsigned char *peer_arena[MAX_TP] = {};
    std::vector<void *> ipc_opened;
    unsigned long long spin_ns = 20ull * 1000000000ull;   // bound on every peer wait (L2B_SPIN_TIMEOUT_MS)
    bool attn_flash = true;                  // flash-decoding attention (false: 3-pass kernel)
    unsigned long long *trace = nullptr;     // L2B_TRACE=1: [launch][TRACE_MAX_CTAS][TRACE_SLOTS] timeline
    int trace_launches = 0;
    int tma_ctas_per_sm = 1;
    int tma_stages = 0;                      // 0 = auto; else forced ring depth
    int tma_prefill = 0;                     // stages in flight before the dependency wait; 0 = the whole ring (L2B_TMA_PREFILL)
    bool big_kernel_tma = true;              // bandwidth-bound GEMVs: TMA-ring kernel (false: register-fed 8-row kernel)
    long long gemv8_min_bytes = 8ll << 20;   // >= this many weight bytes (and n >= big_min_n): streaming kernel; -1 = never
    int big_min_n = 1024;                    // measured r02: at n = 768 the TMA ring (192 of 256 columns per stage) loses to the latency kernel
    int tpr_min_tiles_per_sm = 0;            // > 0: shrink threads-per-row while the grid still has this many tiles per SM (L2B_TPR_TILES)
    int force_kernel = 0;                    // l2b_op_fused_matmul: 0 auto, 1 small, 2 register-fed 8-row, 3 TMA ring
    int launches_per_step = 0;
    std::set<const void *> attr_done;        // kernels whose max-dynamic-smem attribute is set on this device
    // comm (bootstrap / nccl baseline)
    ncclComm_t comm = nullptr;
    // bookkeeping
    int n_appended = 0;
    float last_ms = 0.0f;
    int last_launches = 0;
    double load_ms = 0.0;                    // checkpoint upload wall time (l2b_load_stats)
    uint64_t load_bytes = 0;
    std::string err;
    std::vector<void *> owned;              // device allocations to free
    // upload staging (pinned, double-buffered)
    unsigned char *stage[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    size_t stage_bytes = 0;
    int stage_next = 0;
    // per-kernel profiling (l2b_profile_step)
    bool profiling = false;
    std::vector<cudaEvent_t> prof_ev;
    std::vector<l2b_kernel_time> prof_rec;
};

namespace {

const char *kNoError = "";
thread_local std::string g_create_error;

#define L2B_CUDA(ctx, call)                                                                   \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            char buf__[512];                                                                  \
            snprintf(buf__, sizeof buf__, "%s failed: %s (%s:%d)", #call,                     \
                     cudaGetErrorString(e__), __FILE__, __LINE__);                            \
            (ctx)->err = buf__;                                                               \
            return (e__ == cudaErrorMemoryAllocation) ? L2B_ERR_OOM : L2B_ERR_CUDA;           \
        }                                                                                     \
    } while (0)

#define L2B_NCCL(ctx, call)                                                                   \
    do {                                                                                      \
        ncclResult_t r__ = (call);                                                            \
        if (r__ != ncclSuccess) {                                                             \
            char buf__[512];                                                                  \
            snprintf(buf__, sizeof buf__, "%s failed: %s (%s:%d)", #call,                     \
                     g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "?", __FILE__,      \
                     __LINE__);                                                               \
            (ctx)->err = buf__;                                                               \
            return L2B_ERR_COMM;                                                              \
        }                                                                                     \
    } while (0)

int fail(l2b_ctx *ctx, int code, const char *msg) {
    if (ctx) ctx->err = msg;
    return code;
}

// all ranks this handle drives from this process (1 unless it is an in-process group)
std::vector<l2b_ctx *> locals(l2b_ctx *ctx) {
    if (!ctx->members.empty()) return ctx->members;
    return std::vector<l2b_ctx *>{ctx};
}

template <typename T>
int dev_alloc(l2b_ctx *ctx, T **p, size_t count) {
    void *q = nullptr;
    L2B_CUDA(ctx, cudaMalloc(&q, (count ? count : 1) * sizeof(T)));
    ctx->owned.push_back(q);
    *p = static_cast<T *>(q);
    return L2B_OK;
}

// ---- shape validation (the reference's asserts, src/main.zig:433-434,:534-540,:658-661) ----
int validate_config(const l2b_config *c, int world, std::string *why) {
    auto bad = [&](const char *m) { *why = m; return L2B_ERR_UNSUPPORTED; };
    if (c->dim <= 0 || c->hidden_dim <= 0 || c->n_layers <= 0 || c->n_heads <= 0 ||
        c->n_kv_heads <= 0 || c->vocab_size <= 0 || c->seq_len <= 0) {
        *why = "config fields must be positive";
        return L2B_ERR_INVALID_ARG;
    }
    if (c->dim % c->n_heads) return bad("dim % n_heads != 0");
    if (c->n_heads % c->n_kv_heads) return bad("n_heads % n_kv_heads != 0");
    const int hs = c->dim / c->n_heads;
    if (c->dim % 4 || c->hidden_dim % 4) return bad("dim and hidden_dim must be multiples of 4");
    if (hs % 4) return bad("head_size must be a multiple of 4");
    // the attention kernels write one output element per thread (NT = 256) and the RoPE row of a
    // position is staged as head_size/2 <= 128 pairs
    if (hs > NT) return bad("head_size > 256 is not supported");
    if (world != 1 && world != 2 && world != 4 && world != 8) return bad("world_size must be 1, 2, 4 or 8");
    if (c->n_kv_heads % world) return bad("n_kv_heads % world_size != 0");
    if ((c->hidden_dim / world) % 4 || c->hidden_dim % world) return bad("hidden_dim/world_size must be a multiple of 4");
    if (c->vocab_size % world || (world > 1 && (c->vocab_size / world) % 2)) return bad("vocab_size/world_size must be an even integer");
    return L2B_OK;
}

uint64_t checkpoint_floats(const l2b_config *c) {
    const uint64_t dim = c->dim, hid = c->hidden_dim, L = c->n_layers, V = c->vocab_size, S = c->seq_len;
    const uint64_t hs = dim / c->n_heads, kvd = hs * c->n_kv_heads;
    uint64_t n = V * dim + L * dim + L * dim * dim + 2 * L * dim * kvd + L * dim * dim + L * dim +
                 3 * L * dim * hid + dim + 2 * (S * hs / 2);
    if (!c->shared_weights) n += V * dim;
    return n;
}

// ---- tensor materialisation: upload a (possibly sharded) window, or synthesise it in place ----
enum ShardMode { SH_NONE, SH_ROWS, SH_COLS };
struct Dist { double mean, sigma; float lo, hi; };
constexpr double kSynthInvStd = 2.6428997921303014e-05;  // 1 / sqrt(4*(65536^2-1)/12)

struct Source {
    const float *host = nullptr;   // checkpoint payload or nullptr => synthetic
    uint64_t seed = 0;
};

// Checkpoint ingest (SURVEY 8f.3; the reference slurps the file into pageable heap memory,
// src/main.zig:955-964).  The caller's buffer is pageable, so a plain cudaMemcpy would bounce every
// byte through the driver's small internal staging buffer synchronously.  Here the payload moves
// in chunks through two pinned buffers: while chunk k is in flight on the copy engine, the host
// is already filling the other buffer with chunk k+1 (for column-sharded tensors the host-side
// fill also compacts the strided window, so the DMA is always a dense 1-D copy).
int upload(l2b_ctx *ctx, float *dst, const float *src, uint64_t rows, uint64_t cols, uint64_t src_pitch) {
    if (!ctx->stage[0]) {
        size_t want = 32ull << 20;
        const char *env = getenv("L2B_STAGE_MB");
        if (env && atoi(env) > 0) want = (size_t)atoi(env) << 20;
        ctx->stage_bytes = want;
        for (int i = 0; i < 2; ++i) {
            L2B_CUDA(ctx, cudaHostAlloc((void **)&ctx->stage[i], want, cudaHostAllocDefault));
            L2B_CUDA(ctx, cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
        }
    }
    const uint64_t row_bytes = cols * sizeof(float);
    const bool dense = (src_pitch == cols);
    const uint64_t total = rows * row_bytes;
    uint64_t done = 0;                       // bytes of the dense destination already issued
    while (done < total) {
        const int b = ctx->stage_next;
        ctx->stage_next ^= 1;
        L2B_CUDA(ctx, cudaEventSynchronize(ctx->stage_ev[b]));   // previous DMA out of this buffer finished
        uint64_t chunk = total - done < ctx->stage_bytes ? total - done : ctx->stage_bytes;
        if (!dense) {
            // whole rows only (a chunk never splits a row of a sharded window)
            uint64_t r = chunk / row_bytes;
            if (r == 0) return fail(ctx, L2B_ERR_UNSUPPORTED, "row larger than the upload staging buffer");
            chunk = r * row_bytes;
            const uint64_t row0 = done / row_bytes;
            for (uint64_t i = 0; i < r; ++i)
                memcpy(ctx->stage[b] + i * row_bytes, src + (row0 + i) * src_pitch, row_bytes);
        } else {
            memcpy(ctx->stage[b], reinterpret_cast<const unsigned char *>(src) + done, chunk);
        }
        L2B_CUDA(ctx, cudaMemcpyAsync(reinterpret_cast<unsigned char *>(dst) + done, ctx->stage[b], chunk,
                                      cudaMemcpyHostToDevice, ctx->stream));
        L2B_CUDA(ctx, cudaEventRecord(ctx->stage_ev[b], ctx->stream));
        done += chunk;
    }
    ctx->load_bytes += total;
    return L2B_OK;
}

int materialize(l2b_ctx *ctx, float **dptr, const Source &src, uint64_t payload_off, int tensor_id,
                uint64_t L, uint64_t rows, uint64_t cols, ShardMode mode, Dist dist) {
    const uint64_t g = ctx->world, r = ctx->rank;
    const uint64_t rows_loc = (mode == SH_ROWS) ? rows / g : rows;
    const uint64_t cols_loc = (mode == SH_COLS) ? cols / g : cols;
    const uint64_t row0 = (mode == SH_ROWS) ? r * rows_loc : 0;
    const uint64_t col0 = (mode == SH_COLS) ? r * cols_loc : 0;
    int rc = dev_alloc(ctx, dptr, L * rows_loc * cols_loc);
    if (rc) return rc;
    const uint64_t tensor_seed = mix64(src.seed * 1000003ull + (uint64_t)tensor_id);
    const bool whole = (rows_loc == rows && cols_loc == cols);
    const uint64_t nl = whole ? 1 : L;            // one shot when nothing is cut
    const uint64_t rr = whole ? L * rows : rows_loc;
    for (uint64_t l = 0; l < nl; ++l) {
        float *dst = *dptr + l * rows_loc * cols_loc;
        const uint64_t first = l * rows * cols + row0 * cols + col0;
        if (src.host) {
            rc = upload(ctx, dst, src.host + payload_off + first, rr, cols_loc, cols);
            if (rc) return rc;
        } else {
            const uint64_t total = rr * cols_loc;
            int blocks = (int)((total + 255) / 256 < (uint64_t)(ctx->num_sms * 16)
                                   ? (total + 255) / 256
                                   : (uint64_t)(ctx->num_sms * 16));
            if (blocks < 1) blocks = 1;
            synth_fill_kernel<<<blocks, 256, 0, ctx->stream>>>(dst, rr, cols_loc, first, cols, tensor_seed,
                                                               dist.mean, dist.sigma * kSynthInvStd,
                                                               dist.lo, dist.hi);
            L2B_CUDA(ctx, cudaGetLastError());
        }
    }
    return L2B_OK;
}

// ---- GEMV launch ---------------------------------------------------------------------------
typedef void (*gemv_fn)(const GemvParams);

template <int EPI>
gemv_fn gemv_pick(int tpr) {
    switch (tpr) {
    case 8: return gemv_kernel<8, EPI>;
    case 16: return gemv_kernel<16, EPI>;
    case 32: return gemv_kernel<32, EPI>;
    case 64: return gemv_kernel<64, EPI>;
    case 128: return gemv_kernel<128, EPI>;
    default: return gemv_kernel<256, EPI>;
    }
}
gemv_fn gemv_pick(int epi, int tpr) {
    switch (epi) {
    case EPI_XCHG: return gemv_pick<EPI_XCHG>(tpr);
    case EPI_RESID: return gemv_pick<EPI_RESID>(tpr);
    case EPI_STORE: return gemv_pick<EPI_STORE>(tpr);
    case EPI_ARGMAX: return gemv_pick<EPI_ARGMAX>(tpr);
    case EPI_QKV: return gemv_pick<EPI_QKV>(tpr);
    default: return gemv_pick<EPI_SILU>(tpr);
    }
}

constexpr int kMaxDynSmem = 200 * 1024;
constexpr int kMaxSmemOptin = 227 * 1024 - 2048;   // static __shared__ of the kernels stays under 2 KB

int gemv_tpr(int n) {
    const int n4 = n / 4;
    int tpr = 8;
    while (tpr < 256 && tpr * 2 <= n4 / 2) tpr *= 2;
    return tpr;
}

int prof_mark(l2b_ctx *ctx, const char *name, int layer, uint64_t bytes, cudaStream_t st) {
    if (!ctx->profiling) return L2B_OK;
    cudaEvent_t ev;
    L2B_CUDA(ctx, cudaEventCreate(&ev));
    L2B_CUDA(ctx, cudaEventRecord(ev, st));
    ctx->prof_ev.push_back(ev);
    l2b_kernel_time r{};
    snprintf(r.name, sizeof r.name, "%s", name);
    r.layer = layer;
    r.bytes = bytes;
    ctx->prof_rec.push_back(r);
    return L2B_OK;
}

gemv_fn gemv_tma_pick(int epi) {
    switch (epi) {
    case EPI_XCHG: return gemv_tma_kernel<EPI_XCHG>;
    case EPI_RESID: return gemv_tma_kernel<EPI_RESID>;
    case EPI_STORE: return gemv_tma_kernel<EPI_STORE>;
    case EPI_ARGMAX: return gemv_tma_kernel<EPI_ARGMAX>;
    case EPI_QKV: return gemv_tma_kernel<EPI_QKV>;
    default: return gemv_tma_kernel<EPI_SILU>;
    }
}

gemv_fn gemv8_pick(int epi) {
    switch (epi) {
    case EPI_XCHG: return gemv8_kernel<EPI_XCHG>;
    case EPI_RESID: return gemv8_kernel<EPI_RESID>;
    case EPI_STORE: return gemv8_kernel<EPI_STORE>;
    case EPI_ARGMAX: return gemv8_kernel<EPI_ARGMAX>;
    case EPI_QKV: return gemv8_kernel<EPI_QKV>;
    default: return gemv8_kernel<EPI_SILU>;
    }
}

cudaLaunchAttribute pdl_attr() {
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    return at;
}

unsigned long long *trace_slot(l2b_ctx *ctx) {
    if (!ctx->trace || ctx->profiling) return nullptr;
    return ctx->trace + (size_t)(ctx->last_launches % ctx->trace_launches) * TRACE_MAX_CTAS * TRACE_SLOTS;
}

int launch_gemv(l2b_ctx *ctx, int epi, const GemvParams &p, cudaStream_t st, const char *name = "gemv",
                int layer = -1) {
    {
        int prc = prof_mark(ctx, name, layer, (uint64_t)p.total_rows * p.n * 4ull, st);
        if (prc) return prc;
    }
    const size_t xbytes = (size_t)p.n * 4 * (1 + (p.gamma ? 1 : 0) + (p.parts ? 1 : 0));
    // bandwidth-bound shapes take the TMA-ring kernel (or the register-fed 8-row kernel when
    // L2B_GEMV_BIG=ldg), latency-bound ones the fine-grained kernel
    bool big = ctx->gemv8_min_bytes >= 0 && p.n >= ctx->big_min_n &&
               (uint64_t)p.total_rows * p.n * 4ull >= (uint64_t)ctx->gemv8_min_bytes;
    if (ctx->force_kernel == 1) big = false;
    if (ctx->force_kernel >= 2) big = true;
    // TMA-ring kernel: only x is staged in shared memory, the rest of the SM's 227 KB is the ring
    // (measured: 5-6 stages of 32 KB on ONE CTA per SM beat 2 x 3 stages and beat leaving half
    // the SM to the successor kernel's pre-fill; profiles/r01_tma_ring_variants.md)
    const size_t stage_bytes = (size_t)TMA_STAGE_FLOATS * 4;
    const size_t xonly = (size_t)p.n * 4;
    int nstage = ctx->tma_stages > 0 ? ctx->tma_stages : (int)(((size_t)kMaxSmemOptin - xonly) / stage_bytes);
    if (nstage > TMA_MAX_STAGES) nstage = TMA_MAX_STAGES;
    const bool fused_ok = !p.gamma || p.n <= 5 * (TMA_THREADS - 32) * 4;   // register slices of the rmsnorm gain (MAXV x prologue threads)
    if (p.parts && big) return fail(ctx, L2B_ERR_UNSUPPORTED, "partial-vector prologue is only in the latency kernel");
    bool tma = big && ctx->big_kernel_tma && nstage >= 2 && fused_ok && p.head_size <= 256 &&
               (size_t)nstage * stage_bytes + xonly <= (size_t)kMaxSmemOptin;
    if (ctx->force_kernel == 2) tma = false;
    if (ctx->force_kernel == 3 && !tma) return fail(ctx, L2B_ERR_UNSUPPORTED, "shape does not fit the TMA-ring kernel");
    const size_t smem = tma ? (size_t)nstage * stage_bytes + xonly : xbytes;
    if (smem > (size_t)kMaxSmemOptin) return fail(ctx, L2B_ERR_UNSUPPORTED, "activation vector too large for shared memory");
    int tpr = gemv_tpr(p.n);
    // many-row matrices (the classifier): fewer threads per row = more 128-bit loads in flight per
    // thread and fewer shuffle steps per row, as long as the grid still covers the SMs
    while (ctx->tpr_min_tiles_per_sm > 0 && tpr > 8 &&
           (p.total_rows + (NT / (tpr / 2)) * GEMV_R - 1) / ((NT / (tpr / 2)) * GEMV_R) >= ctx->tpr_min_tiles_per_sm * ctx->num_sms)
        tpr /= 2;
    gemv_fn fn = tma ? gemv_tma_pick(epi) : big ? gemv8_pick(epi) : gemv_pick(epi, tpr);
    if (!ctx->attr_done.count((const void *)fn)) {
        L2B_CUDA(ctx, cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmemOptin));
        ctx->attr_done.insert((const void *)fn);
    }
    const int threads = tma ? TMA_THREADS : NT;
    int occ = 0;
    L2B_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, threads, smem));
    if (occ < 1) occ = 1;
    if (tma && occ > ctx->tma_ctas_per_sm) occ = ctx->tma_ctas_per_sm;   // leave room for the next kernel's CTA
    int grid = ctx->num_sms * occ;
    if (big) {
        const int npairs = (p.total_rows + 1) / 2;
        if (grid > npairs) grid = npairs;
    } else {
        const int tile_rows = (NT / tpr) * GEMV_R;
        const int ntiles = (p.total_rows + tile_rows - 1) / tile_rows;
        if (grid > ntiles) grid = ntiles;
    }
    if (grid < 1) grid = 1;
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(threads);
    lc.dynamicSmemBytes = smem;
    lc.stream = st;
    cudaLaunchAttribute at[1] = {pdl_attr()};
    lc.attrs = at;
    lc.numAttrs = ctx->use_pdl ? 1 : 0;
    GemvParams pp = p;
    pp.nstage = nstage;
    pp.nprefill = (ctx->tma_prefill > 0 && ctx->tma_prefill < nstage) ? ctx->tma_prefill : nstage;
    pp.spin_ns = ctx->spin_ns;
    pp.trace = trace_slot(ctx);
    ctx->last_grid = grid;
    L2B_CUDA(ctx, cudaLaunchKernelEx(&lc, fn, pp));
    ++ctx->last_launches;
    return L2B_OK;
}

// flash-decoding form when head_size/4 splits into 1..8 float4 per lane, else the 3-pass kernel
typedef void (*attn_fn)(const AttnParams);
attn_fn pick_attention(int head_size, bool flash, size_t *smem) {
    const int hs4 = head_size / 4;
    const int lpr = (hs4 % 8 == 0) ? 8 : (hs4 % 4 == 0) ? 4 : (hs4 % 2 == 0) ? 2 : 1;
    const int nf = hs4 / lpr;
    attn_fn f2 = nullptr;
    if (flash) {
        switch (nf) {
        case 1: f2 = attention_flash_kernel<1>; break;
        case 2: f2 = attention_flash_kernel<2>; break;
        case 3: f2 = attention_flash_kernel<3>; break;
        case 4: f2 = attention_flash_kernel<4>; break;
        case 5: f2 = attention_flash_kernel<5>; break;
        case 6: f2 = attention_flash_kernel<6>; break;
        case 8: f2 = attention_flash_kernel<8>; break;
        default: break;
        }
    }
    if (!f2) return attention_kernel;
    const int ng = NWARP * (32 / lpr);
    *smem = ((size_t)ng * head_size + 3 * (size_t)ng) * sizeof(float);
    return f2;
}

typedef void (*attn_wo_fn)(const AttnWoParams);
attn_wo_fn pick_attn_wo(int head_size, size_t *smem) {
    const int hs4 = head_size / 4;
    const int lpr = (hs4 % 8 == 0) ? 8 : (hs4 % 4 == 0) ? 4 : (hs4 % 2 == 0) ? 2 : 1;
    const int nf = hs4 / lpr;
    const int ng = NWARP * (32 / lpr);
    *smem = ((size_t)ng * head_size + 3 * (size_t)ng + 2 * (size_t)head_size + 4) * sizeof(float);
    switch (nf) {
    case 1: return attn_wo_kernel<1>;
    case 2: return attn_wo_kernel<2>;
    case 3: return attn_wo_kernel<3>;
    case 4: return attn_wo_kernel<4>;
    case 5: return attn_wo_kernel<5>;
    case 6: return attn_wo_kernel<6>;
    case 8: return attn_wo_kernel<8>;
    default: return nullptr;
    }
}

// attention + wo of one layer in one cluster launch (small models): partial vectors -> ctx->attn_parts
int launch_attn_wo(l2b_ctx *ctx, int layer, cudaStream_t st) {
    if (ctx->profiling) {
        const int hpos = ctx->n_appended > 0 ? ctx->n_appended - 1 : 0;
        int prc = prof_mark(ctx, "attn_wo", layer, 2ull * (uint64_t)(hpos + 1) * ctx->kv_loc * 4ull + (uint64_t)ctx->dim * ctx->q_loc * 4ull, st);
        if (prc) return prc;
    }
    AttnWoParams q{};
    AttnParams &a = q.a;
    a.ctl = ctx->ctl;
    a.q = ctx->q;
    const size_t loff = (size_t)layer * ctx->cfg.seq_len * ctx->kv_loc;   // :354
    a.kcache = ctx->kcache + loff;
    a.vcache = ctx->vcache + loff;
    a.head_size = ctx->head_size;
    a.kv_dim = ctx->kv_loc;
    a.kv_mul = ctx->kv_mul;
    a.trace = nullptr;
    q.wo = ctx->wo + (size_t)layer * ctx->dim * ctx->q_loc;
    q.parts = ctx->attn_parts;
    q.dim = ctx->dim;
    q.q_dim = ctx->q_loc;
    size_t smem = 0;
    attn_wo_fn fn = pick_attn_wo(ctx->head_size, &smem);
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(ctx->heads_loc, ctx->attn_R);
    lc.blockDim = dim3(NT);
    lc.dynamicSmemBytes = smem;
    lc.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 1; at[0].val.clusterDim.y = ctx->attn_R; at[0].val.clusterDim.z = 1;
    at[1] = pdl_attr();
    lc.attrs = at;
    lc.numAttrs = ctx->use_pdl ? 2 : 1;
    L2B_CUDA(ctx, cudaLaunchKernelEx(&lc, fn, q));
    ++ctx->last_launches;
    return L2B_OK;
}

int launch_attention(l2b_ctx *ctx, int layer, cudaStream_t st) {
    if (ctx->profiling) {
        const int hpos = ctx->n_appended > 0 ? ctx->n_appended - 1 : 0;
        int prc = prof_mark(ctx, "attention", layer, 2ull * (uint64_t)(hpos + 1) * ctx->kv_loc * 4ull, st);
        if (prc) return prc;
    }
    AttnParams a{};
    a.ctl = ctx->ctl;
    a.q = ctx->q;
    const size_t loff = (size_t)layer * ctx->cfg.seq_len * ctx->kv_loc;   // :354
    a.kcache = ctx->kcache + loff;
    a.vcache = ctx->vcache + loff;
    a.xb = ctx->xb;
    a.part_o = ctx->part_o;
    a.part_ml = ctx->part_ml;
    a.counters = ctx->counters;
    a.head_size = ctx->head_size;
    a.kv_dim = ctx->kv_loc;
    a.kv_mul = ctx->kv_mul;
    a.nsplit = ctx->nsplit;
    a.min_chunk = ctx->min_chunk;
    a.vec = nullptr;                 // single position from the control block
    a.seq_len = ctx->cfg.seq_len;
    a.trace = trace_slot(ctx);
    size_t smem = ctx->attn_smem;
    attn_fn fn = pick_attention(ctx->head_size, ctx->attn_flash, &smem);
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(ctx->heads_loc, ctx->nsplit);
    lc.blockDim = dim3(NT);
    lc.dynamicSmemBytes = smem;
    lc.stream = st;
    cudaLaunchAttribute at[1] = {pdl_attr()};
    lc.attrs = at;
    lc.numAttrs = ctx->use_pdl ? 1 : 0;
    L2B_CUDA(ctx, cudaLaunchKernelEx(&lc, fn, a));
    ++ctx->last_launches;
    return L2B_OK;
}

// ---- tensor-parallel landing areas (offsets into an arena; same layout on every rank) --------
unsigned long long *ll_red_at(unsigned char *arena, const l2b_ctx *c, int slot, int src_rank) {
    return reinterpret_cast<unsigned long long *>(arena + c->off_red) + ((size_t)slot * c->world + src_rank) * c->dim;
}
unsigned long long *ll_logits_at(unsigned char *arena, const l2b_ctx *c) {
    return reinterpret_cast<unsigned long long *>(arena + c->off_logits);
}
unsigned long long *ll_amax_at(unsigned char *arena, const l2b_ctx *c, int src_rank) {
    return reinterpret_cast<unsigned long long *>(arena + c->off_amax) + 2 * (size_t)src_rank;
}


int launch_small(l2b_ctx *ctx, const void *fn, dim3 grid, dim3 block, void **args, cudaStream_t st, bool pdl) {
    cudaLaunchConfig_t lc{};
    lc.gridDim = grid;
    lc.blockDim = block;
    lc.stream = st;
    cudaLaunchAttribute at[1] = {pdl_attr()};
    lc.attrs = at;
    lc.numAttrs = (pdl && ctx->use_pdl) ? 1 : 0;
    L2B_CUDA(ctx, cudaLaunchKernelExC(&lc, fn, args));
    ++ctx->last_launches;
    return L2B_OK;
}

int launch_advance(l2b_ctx *ctx, cudaStream_t st, bool forced, bool exchange) {
    AdvanceParams a{};
    a.ctl = ctx->ctl;
    a.amax = ctx->amax;
    a.forced = forced ? ctx->gen_forced : nullptr;
    a.out_next = ctx->gen_out;
    a.n_done = ctx->gen_ndone;
    a.world = exchange ? ctx->world : 1;
    a.rank = ctx->rank;
    a.spin_ns = ctx->spin_ns;
    if (exchange) {
        for (int r = 0; r < ctx->world; ++r) a.ll_out[r] = ll_amax_at(ctx->peer_arena[r], ctx, ctx->rank);
        a.ll_in = ll_amax_at(ctx->arena, ctx, 0);
    }
    void *args[] = {&a};
    return launch_small(ctx, (const void *)advance_kernel, dim3(1), dim3(32), args, st, true);
}

// One decode step on `st` (transformer(), src/main.zig:285-430).  All (token, pos) dependence is
// through ctx->ctl, so the sequence is capturable once and replayed.
int enqueue_step(l2b_ctx *ctx, cudaStream_t st, StepMode mode) {
    const l2b_config &c = ctx->cfg;
    const int dim = ctx->dim;
    const bool tp = ctx->world > 1;
    const bool p2p = tp && ctx->use_p2p;
    // my partial rows go to every rank; slice owners then fold all ranks' rows into x (tp_reduce_tail)
    auto produce_slot = [&](GemvParams &g, int slot, float *x) {
        g.ll_ndst = ctx->world;
        for (int r = 0; r < ctx->world; ++r) g.ll_out[r] = ll_red_at(ctx->peer_arena[r], ctx, slot, ctx->rank);
        g.ll_in = ll_red_at(ctx->arena, ctx, slot, 0);
        g.xres = x;
        g.xworld = ctx->world;
    };
    // wo / w2: row-parallel GEMV whose result is added to the residual stream (:392-395, :419-422)
    auto residual_gemv = [&](GemvParams &g, float *x, int slot, const char *name, int l) -> int {
        g.total_rows = dim; g.rows0 = dim;
        int rc;
        if (!tp) {
            g.out0 = x;
            rc = launch_gemv(ctx, EPI_RESID, g, st, name, l);
        } else if (p2p) {
            produce_slot(g, slot, x);
            rc = launch_gemv(ctx, EPI_XCHG, g, st, name, l);
        } else {
            g.out0 = ctx->delta;
            rc = launch_gemv(ctx, EPI_STORE, g, st, name, l);
            if (rc) return rc;
            L2B_NCCL(ctx, g_nccl.AllReduce(ctx->delta, ctx->delta, dim, ncclFloat, ncclSum, ctx->comm, st));
            resid_add_kernel<<<(dim + NT - 1) / NT, NT, 0, st>>>(x, ctx->delta, dim, ctx->ctl);
            L2B_CUDA(ctx, cudaGetLastError());
            ++ctx->last_launches;
        }
        return rc;
    };
    // small-model fusion (world == 1): attention+wo leaves its result as one partial vector per head
    // that the NEXT kernel's prologue sums into x; such a kernel reads x from one buffer and CTA 0
    // writes the new x to the other (ping-pong), everything else updates x in place
    float *Xc = ctx->X, *Xo = ctx->Xalt;
    const float *pend = nullptr;             // partial vectors still to be folded into x
    int npend = 0;

    auto fold_pending = [&](GemvParams &g) {
        g.x_in = Xc;
        if (pend) {
            g.parts = pend; g.nparts = npend; g.x_out = Xo;
            float *t = Xc; Xc = Xo; Xo = t;
            pend = nullptr; npend = 0;
        }
    };
    for (int l = 0; l < c.n_layers; ++l) {
        // ---- rmsnorm + q,k,v + RoPE + KV append (:305-358)
        GemvParams p{};
        p.ctl = ctx->ctl;
        p.n = dim;
        fold_pending(p);
        if (l == 0) {
            p.emb = ctx->emb;                 // :295-296
            p.x_out = Xc;
            p.bump_epoch = 1;
        }
        p.gamma = ctx->rms_att + (size_t)l * dim;
        p.w0 = ctx->wq + (size_t)l * ctx->q_loc * dim;
        p.w1 = ctx->wk + (size_t)l * ctx->kv_loc * dim;
        p.w2 = ctx->wv + (size_t)l * ctx->kv_loc * dim;
        p.rows0 = ctx->q_loc; p.rows1 = ctx->kv_loc; p.rows2 = ctx->kv_loc;
        p.total_rows = ctx->q_loc + 2 * ctx->kv_loc;
        p.out0 = ctx->q;
        const size_t loff = (size_t)l * c.seq_len * ctx->kv_loc;
        p.kcache = ctx->kcache + loff;
        p.vcache = ctx->vcache + loff;
        p.rope_cos = ctx->rope_cos; p.rope_sin = ctx->rope_sin;
        p.head_size = ctx->head_size; p.kv_dim = ctx->kv_loc;
        int rc = launch_gemv(ctx, EPI_QKV, p, st, "qkv_rope", l);
        if (rc) return rc;

        if (ctx->fuse_attn) {
            // ---- attention + wo in one cluster launch (:361-392); the add of :395 happens in the next prologue
            rc = launch_attn_wo(ctx, l, st);
            if (rc) return rc;
            pend = ctx->attn_parts; npend = ctx->heads_loc;
        } else {
            // ---- attention (:361-389)
            rc = launch_attention(ctx, l, st);
            if (rc) return rc;
            // ---- wo + residual (:392-395)
            GemvParams o{};
            o.ctl = ctx->ctl;
            o.n = ctx->q_loc;
            o.x_in = ctx->xb;
            o.w0 = ctx->wo + (size_t)l * dim * ctx->q_loc;
            rc = residual_gemv(o, Xc, 2 * l, "wo", l);
            if (rc) return rc;
        }

        // ---- rmsnorm + w1,w3 + SiLU*mul (:398-416)
        GemvParams f{};
        f.ctl = ctx->ctl;
        f.n = dim;
        fold_pending(f);
        f.gamma = ctx->rms_ffn + (size_t)l * dim;
        f.w0 = ctx->w1 + (size_t)l * ctx->hid_loc * dim;
        f.w1 = ctx->w3 + (size_t)l * ctx->hid_loc * dim;
        f.rows0 = ctx->hid_loc;
        f.total_rows = 2 * ctx->hid_loc;
        f.out0 = ctx->hb;
        rc = launch_gemv(ctx, EPI_SILU, f, st, "w13_silu", l);
        if (rc) return rc;

        // ---- w2 + residual (:419-422)
        GemvParams d{};
        d.ctl = ctx->ctl;
        d.n = ctx->hid_loc;
        d.x_in = ctx->hb;
        d.w0 = ctx->w2 + (size_t)l * dim * ctx->hid_loc;
        rc = residual_gemv(d, Xc, 2 * l + 1, "w2", l);
        if (rc) return rc;
    }
    if (mode == MODE_NOCLS) {   // prompt prefill: the logits of this position are never looked at (:996-1000)
        ctx->final_X = Xc;
        return L2B_OK;
    }
    // ---- final rmsnorm + classifier (:426-429)
    GemvParams k{};
    k.ctl = ctx->ctl;
    k.n = dim;
    fold_pending(k);
    ctx->final_X = Xc;
    k.gamma = ctx->rms_final;
    k.w0 = ctx->wcls;
    k.total_rows = ctx->vocab_loc; k.rows0 = ctx->vocab_loc;
    k.out0 = tp ? ctx->logits_loc : ctx->logits;
    k.amax = ctx->amax;
    k.row_base = ctx->rank * ctx->vocab_loc;
    const bool want_argmax = (mode == MODE_ARGMAX);
    int epi = want_argmax ? EPI_ARGMAX : EPI_STORE;
    const bool in_process = ctx->leader != nullptr;
    if (p2p && !want_argmax) {
        // logits slices travel as LL units: to every rank (one process per GPU: each rank's caller gets
        // the logits), or to rank 0 only (in-process group: one caller)
        epi = EPI_XCHG;
        if (in_process) {
            k.ll_ndst = 1;
            k.ll_out[0] = ll_logits_at(ctx->peer_arena[0], ctx);
        } else {
            k.ll_ndst = ctx->world;
            for (int r = 0; r < ctx->world; ++r) k.ll_out[r] = ll_logits_at(ctx->peer_arena[r], ctx);
        }
    }
    int rc = launch_gemv(ctx, epi, k, st, "classifier", -1);
    if (rc) return rc;
    if (tp) {
        if (p2p) {
            if (!want_argmax && (!in_process || ctx->rank == 0)) {
                float *lg = ctx->logits;
                const unsigned long long *in = ll_logits_at(ctx->arena, ctx);
                int V = c.vocab_size;
                const int *ctl = ctx->ctl;
                unsigned long long spin = ctx->spin_ns;
                void *args[] = {&lg, &in, &V, &ctl, &spin};
                int blocks = (V / 2 + NT - 1) / NT;
                if (blocks > ctx->num_sms) blocks = ctx->num_sms;
                rc = launch_small(ctx, (const void *)gather_logits_kernel, dim3(blocks), dim3(NT), args, st, true);
                if (rc) return rc;
            }
        } else if (want_argmax) {
            L2B_NCCL(ctx, g_nccl.AllReduce(ctx->amax, ctx->amax, 1, ncclUint64, ncclMax, ctx->comm, st));
        } else {
            L2B_NCCL(ctx, g_nccl.AllGather(ctx->logits_loc, ctx->logits, ctx->vocab_loc, ncclFloat, ctx->comm, st));
        }
    }
    return L2B_OK;
}

int launch_sample_prep(l2b_ctx *ctx, cudaStream_t st) {
    float *lg = ctx->logits;
    int V = ctx->cfg.vocab_size;
    const int *ctl = ctx->ctl;
    ProbIndex *cand = ctx->cand;
    int cap = kCandCap;
    int *n_cand = ctx->n_cand;
    void *args[] = {&lg, &V, &ctl, &cand, &cap, &n_cand};
    return launch_small(ctx, (const void *)sample_prep_kernel, dim3(1), dim3(SAMP_THREADS), args, st, true);
}

// everything one call needs, as it is captured into (or eagerly enqueued instead of) graph `which`
int enqueue_call(l2b_ctx *ctx, cudaStream_t st, int which) {
    const bool sink = !ctx->leader || ctx->rank == 0;   // in-process group: only rank 0 returns data to the host
    const bool loop = (which == G_ARGMAX_LOOP || which == G_PREFILL_LOOP);   // (token, pos) advance on the device
    if (!loop)
        L2B_CUDA(ctx, cudaMemcpyAsync(ctx->ctl, ctx->h_ctl, CTL_HOST_WORDS * sizeof(int), cudaMemcpyHostToDevice, st));
    const StepMode mode = (which == G_LOGITS) ? MODE_LOGITS : (which == G_SAMPLE) ? MODE_SAMPLE
                          : (which == G_PREFILL_LOOP) ? MODE_NOCLS : MODE_ARGMAX;
    int rc = enqueue_step(ctx, st, mode);
    if (rc) return rc;
    const size_t vbytes = (size_t)ctx->cfg.vocab_size * sizeof(float);
    switch (which) {
    case G_LOGITS:
        if (sink) L2B_CUDA(ctx, cudaMemcpyAsync(ctx->h_logits, ctx->logits, vbytes, cudaMemcpyDeviceToHost, st));
        break;
    case G_SAMPLE:
        if (sink) {
            rc = launch_sample_prep(ctx, st);
            if (rc) return rc;
            L2B_CUDA(ctx, cudaMemcpyAsync(ctx->h_logits, ctx->logits, vbytes, cudaMemcpyDeviceToHost, st));
            L2B_CUDA(ctx, cudaMemcpyAsync(ctx->h_cand, ctx->cand, (size_t)kCandCap * sizeof(ProbIndex), cudaMemcpyDeviceToHost, st));
            L2B_CUDA(ctx, cudaMemcpyAsync(ctx->h_ints + 2, ctx->n_cand, sizeof(int), cudaMemcpyDeviceToHost, st));
        }
        break;
    case G_ARGMAX_ONE:
        rc = launch_advance(ctx, st, false, ctx->world > 1 && ctx->use_p2p);
        if (rc) return rc;
        if (sink) L2B_CUDA(ctx, cudaMemcpyAsync(ctx->h_ints, ctx->gen_out, sizeof(int), cudaMemcpyDeviceToHost, st));
        break;
    case G_PREFILL_LOOP:   // every next token is forced: no argmax to exchange
        rc = launch_advance(ctx, st, true, false);
        if (rc) return rc;
        break;
    default:   // G_ARGMAX_LOOP
        rc = launch_advance(ctx, st, true, ctx->world > 1 && ctx->use_p2p);
        if (rc) return rc;
        break;
    }
    if (!loop && ctx->world > 1)   // the error word can only be raised by a tensor-parallel peer wait
        L2B_CUDA(ctx, cudaMemcpyAsync(ctx->h_ctl + CTL_WORDS, ctx->ctl, CTL_WORDS * sizeof(int), cudaMemcpyDeviceToHost, st));
    return L2B_OK;
}

int build_graphs(l2b_ctx *ctx) {
    for (int which = 0; which < G_COUNT; ++which) {
        cudaGraph_t g = nullptr;
        L2B_CUDA(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed));
        ctx->last_launches = 0;
        int rc = enqueue_call(ctx, ctx->stream, which);
        cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
        if (rc) { if (g) cudaGraphDestroy(g); return rc; }
        L2B_CUDA(ctx, e);
        L2B_CUDA(ctx, cudaGraphInstantiate(&ctx->graphs[which], g, 0));
        L2B_CUDA(ctx, cudaGraphDestroy(g));
        if (which == G_LOGITS) ctx->launches_per_step = ctx->last_launches;
    }
    return L2B_OK;
}

int check_step_args(l2b_ctx *ctx, int token, int pos) {
    if (!ctx) return L2B_ERR_INVALID_ARG;
    if (token < 0 || token >= ctx->cfg.vocab_size) return fail(ctx, L2B_ERR_INVALID_ARG, "token out of range");
    if (pos < 0 || pos >= ctx->cfg.seq_len) return fail(ctx, L2B_ERR_INVALID_ARG, "pos out of range");
    if (pos > ctx->n_appended) return fail(ctx, L2B_ERR_STATE, "pos skips ahead of the KV cache");
    return L2B_OK;
}

#define L2B_TRY(expr)                                  \
    do {                                               \
        int rc__ = (expr);                             \
        if (rc__) {                                    \
            g_create_error = ctx->err;                 \
            return rc__;                               \
        }                                              \
    } while (0)

int cuda_try(l2b_ctx *ctx, cudaError_t e, const char *what) {
    if (e == cudaSuccess) return L2B_OK;
    ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? L2B_ERR_OOM : L2B_ERR_CUDA;
}

// Load every kernel this library can launch onto the current device NOW.  With CUDA's default lazy
// module loading a kernel is loaded at its first launch, which can need the device to go idle —
// and a tensor-parallel kernel that is spinning on a peer (which the same host thread has not
// launched yet, in-process groups) would then never let it.
int preload_kernels(l2b_ctx *ctx) {
    cudaFuncAttributes fa;
    const int tprs[] = {8, 16, 32, 64, 128, 256};
    for (int epi = 0; epi < EPI_COUNT; ++epi) {
        for (int tpr : tprs) L2B_CUDA(ctx, cudaFuncGetAttributes(&fa, (const void *)gemv_pick(epi, tpr)));
        L2B_CUDA(ctx, cudaFuncGetAttributes(&fa, (const void *)gemv8_pick(epi)));
        L2B_CUDA(ctx, cudaFuncGetAttributes(&fa, (const void *)gemv_tma_pick(epi)));
    }
    size_t smem = 0;
    L2B_CUDA(ctx, cudaFuncGetAttributes(&fa, (const void *)pick_attention(ctx->head_size, true, &smem)));
    if (pick_attn_wo(ctx->head_size, &smem)) L2B_CUDA(ctx, cudaFuncGetAttributes(&fa, (const void *)pick_attn_wo(ctx->head_size, &smem)));
    const void *others[] = {(const void *)attention_kernel, (const void *)advance_kernel, (const void *)advance_batch_kernel,
                            (const void *)gather_logits_kernel,
                            (const void *)resid_add_kernel, (const void *)sample_prep_kernel, (const void *)synth_fill_kernel};
    for (const void *f : others) L2B_CUDA(ctx, cudaFuncGetAttributes(&fa, f));
    return L2B_OK;
}

// ---- creation, stage 1: weights + run state of one rank (no peer is touched) ------------------
// shape of one rank's shard, and the device objects every context needs
int open_rank(l2b_ctx *ctx, const l2b_config *cfg, int rank, int world, int device, int num_sms) {
    ctx->cfg = *cfg;
    ctx->rank = rank; ctx->world = world; ctx->device = device;
    ctx->num_sms = num_sms;
    ctx->dim = cfg->dim; ctx->hidden = cfg->hidden_dim;
    ctx->head_size = cfg->dim / cfg->n_heads;
    ctx->kv_mul = cfg->n_heads / cfg->n_kv_heads;
    ctx->q_dim = cfg->dim;
    ctx->kv_dim = ctx->head_size * cfg->n_kv_heads;
    ctx->q_loc = ctx->q_dim / world; ctx->kv_loc = ctx->kv_dim / world;
    ctx->hid_loc = cfg->hidden_dim / world;
    ctx->heads_loc = cfg->n_heads / world;
    ctx->vocab_loc = cfg->vocab_size / world;

    L2B_TRY(cuda_try(ctx, cudaSetDevice(device), "cudaSetDevice"));
    L2B_TRY(cuda_try(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking), "cudaStreamCreate"));
    L2B_TRY(cuda_try(ctx, cudaEventCreate(&ctx->ev0), "cudaEventCreate"));
    L2B_TRY(cuda_try(ctx, cudaEventCreate(&ctx->ev1), "cudaEventCreate"));
    L2B_TRY(preload_kernels(ctx));
    return L2B_OK;
}

int init_run_state(l2b_ctx *ctx, const float *rope_cos, const float *rope_sin, const l2b_ctx *rope_from);

int create_rank(l2b_ctx *ctx, const l2b_config *cfg, const Source &src, const float *rope_cos,
                const float *rope_sin, int rank, int world, int device) {
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { ctx->err = "cudaGetDeviceProperties failed"; g_create_error = ctx->err; return L2B_ERR_CUDA; }
    if (prop.major != 10) { ctx->err = "device is not compute capability 10.x (built for sm_100a only)"; g_create_error = ctx->err; return L2B_ERR_NO_DEVICE; }
    L2B_TRY(open_rank(ctx, cfg, rank, world, device, prop.multiProcessorCount));

    const uint64_t dim = cfg->dim, hid = cfg->hidden_dim, L = cfg->n_layers, V = cfg->vocab_size, S = cfg->seq_len;
    const uint64_t hs = ctx->head_size, kvd = ctx->kv_dim;
    const double sd = sqrt(288.0 / (double)dim), sh = sqrt(768.0 / (double)hid);
    const float BIG = 3.0e38f;
    // payload offsets in checkpoint order (src/main.zig:85-112)
    uint64_t off = 0;
    const uint64_t o_emb = off;  off += V * dim;
    const uint64_t o_ratt = off; off += L * dim;
    const uint64_t o_wq = off;   off += L * dim * dim;
    const uint64_t o_wk = off;   off += L * kvd * dim;
    const uint64_t o_wv = off;   off += L * kvd * dim;
    const uint64_t o_wo = off;   off += L * dim * dim;
    const uint64_t o_rffn = off; off += L * dim;
    const uint64_t o_w1 = off;   off += L * hid * dim;
    const uint64_t o_w2 = off;   off += L * dim * hid;
    const uint64_t o_w3 = off;   off += L * hid * dim;
    const uint64_t o_rfin = off; off += dim;
    off += 2 * (S * hs / 2);     // freq_cis_real/imag: not used by transformer() (:67-69, :298-300)
    const uint64_t o_wcls = off;

    const auto t_load0 = std::chrono::steady_clock::now();
    L2B_TRY(materialize(ctx, &ctx->emb, src, o_emb, 1, 1, V, dim, SH_NONE, {0.0, 0.04, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->rms_att, src, o_ratt, 2, 1, L, dim, SH_NONE, {1.35, 0.35, 0.25f, 2.4f}));
    L2B_TRY(materialize(ctx, &ctx->wq, src, o_wq, 3, L, dim, dim, SH_ROWS, {0.0, 0.04 * sd, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->wk, src, o_wk, 4, L, kvd, dim, SH_ROWS, {0.0, 0.04 * sd, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->wv, src, o_wv, 5, L, kvd, dim, SH_ROWS, {0.0, 0.02 * sd, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->wo, src, o_wo, 6, L, dim, dim, SH_COLS, {0.0, 0.02 * sd, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->rms_ffn, src, o_rffn, 7, 1, L, dim, SH_NONE, {1.35, 0.35, 0.25f, 2.4f}));
    L2B_TRY(materialize(ctx, &ctx->w1, src, o_w1, 8, L, hid, dim, SH_ROWS, {0.0, 0.026 * sd, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->w2, src, o_w2, 9, L, dim, hid, SH_COLS, {0.0, 0.026 * sh, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->w3, src, o_w3, 10, L, hid, dim, SH_ROWS, {0.0, 0.026 * sd, -BIG, BIG}));
    L2B_TRY(materialize(ctx, &ctx->rms_final, src, o_rfin, 11, 1, 1, dim, SH_NONE, {7.1, 0.6, 3.0f, 10.0f}));
    if (cfg->shared_weights) {
        ctx->wcls = ctx->emb + (size_t)rank * ctx->vocab_loc * dim;   // :112
    } else {
        L2B_TRY(materialize(ctx, &ctx->wcls, src, o_wcls, 14, 1, V, dim, SH_ROWS, {0.0, 0.04, -BIG, BIG}));
    }
    L2B_TRY(cuda_try(ctx, cudaStreamSynchronize(ctx->stream), "weight upload"));
    ctx->load_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_load0).count();
    for (int i = 0; i < 2; ++i) {          // the staging buffers are only needed during the upload
        if (ctx->stage[i]) { cudaFreeHost(ctx->stage[i]); ctx->stage[i] = nullptr; }
        if (ctx->stage_ev[i]) { cudaEventDestroy(ctx->stage_ev[i]); ctx->stage_ev[i] = nullptr; }
    }
    // everything allocated so far is a weight tensor: it moves to the store that streams share
    ctx->weights = std::make_shared<WeightStore>();
    ctx->weights->device = device;
    ctx->weights->owned.swap(ctx->owned);
    return init_run_state(ctx, rope_cos, rope_sin, nullptr);
}

// ---- run state of one context (RunState.init, :137-154): its KV cache, buffers, graphs' inputs.
// rope_from != nullptr: copy that context's RoPE table (a stream over its weights)
int init_run_state(l2b_ctx *ctx, const float *rope_cos, const float *rope_sin, const l2b_ctx *rope_from) {
    const l2b_config *cfg = &ctx->cfg;
    const int world = ctx->world, rank = ctx->rank;
    const uint64_t dim = cfg->dim, L = cfg->n_layers, V = cfg->vocab_size, S = cfg->seq_len;
    const uint64_t hs = ctx->head_size;
    L2B_TRY(dev_alloc(ctx, &ctx->X, dim));
    L2B_TRY(dev_alloc(ctx, &ctx->Xalt, dim));
    {
        // small-model fusion (measured on B200, profiles/r02_small_models.md): attention + wo as one
        // cluster kernel (8 CTAs per head) is +7 % on stories15M (31 -> 25 kernels per token) and -1 % on
        // stories110M, so it is on for dim <= 512 only (L2B_FUSE=0|1 overrides)
        const char *ef = getenv("L2B_FUSE");
        const int want = ef ? atoi(ef) : (dim <= 512 ? 1 : 0);
        size_t smem_aw = 0;
        ctx->fuse_attn = (want & 1) && world == 1 && dim < 1024 && pick_attn_wo((int)hs, &smem_aw) != nullptr;
        const char *er = getenv("L2B_ATTN_R");
        ctx->attn_R = er && atoi(er) >= 1 && atoi(er) <= 8 ? atoi(er) : 8;
        if (ctx->fuse_attn) L2B_TRY(dev_alloc(ctx, &ctx->attn_parts, (size_t)cfg->n_heads * dim));
    }
    L2B_TRY(dev_alloc(ctx, &ctx->delta, dim));
    L2B_TRY(dev_alloc(ctx, &ctx->q, (size_t)ctx->q_loc));
    L2B_TRY(dev_alloc(ctx, &ctx->xb, (size_t)ctx->q_loc));
    L2B_TRY(dev_alloc(ctx, &ctx->hb, (size_t)ctx->hid_loc));
    L2B_TRY(dev_alloc(ctx, &ctx->logits, V));
    if (world > 1) L2B_TRY(dev_alloc(ctx, &ctx->logits_loc, (size_t)ctx->vocab_loc));
    L2B_TRY(dev_alloc(ctx, &ctx->kcache, L * S * ctx->kv_loc));
    L2B_TRY(dev_alloc(ctx, &ctx->vcache, L * S * ctx->kv_loc));
    L2B_TRY(dev_alloc(ctx, &ctx->rope_cos, S * hs / 2));
    L2B_TRY(dev_alloc(ctx, &ctx->rope_sin, S * hs / 2));
    L2B_TRY(dev_alloc(ctx, &ctx->ctl, (size_t)CTL_WORDS));
    L2B_TRY(dev_alloc(ctx, &ctx->amax, (size_t)1));
    L2B_TRY(dev_alloc(ctx, &ctx->gen_forced, S));
    L2B_TRY(dev_alloc(ctx, &ctx->gen_out, S));
    L2B_TRY(dev_alloc(ctx, &ctx->gen_ndone, (size_t)1));
    L2B_TRY(dev_alloc(ctx, &ctx->cand, (size_t)kCandCap));
    L2B_TRY(dev_alloc(ctx, &ctx->n_cand, (size_t)1));
    L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->ctl, 0, CTL_WORDS * sizeof(int), ctx->stream), "memset"));
    L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->X, 0, dim * sizeof(float), ctx->stream), "memset"));
    L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->amax, 0, sizeof(unsigned long long), ctx->stream), "memset"));
    L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->gen_forced, 0xff, S * sizeof(int), ctx->stream), "memset"));
    L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->kcache, 0, L * S * ctx->kv_loc * sizeof(float), ctx->stream), "memset"));
    L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->vcache, 0, L * S * ctx->kv_loc * sizeof(float), ctx->stream), "memset"));

    // ---- attention launch shape: enough (head, split) CTAs to cover the SMs, chunks >= min_chunk positions
    {
        const char *envc = getenv("L2B_ATTN_MIN_CHUNK");
        if (envc && atoi(envc) >= 8) ctx->min_chunk = atoi(envc);
        int ns = (2 * ctx->num_sms + ctx->heads_loc - 1) / ctx->heads_loc;
        const int max_by_len = (int)((S + ctx->min_chunk - 1) / ctx->min_chunk);
        if (ns > max_by_len) ns = max_by_len;
        if (ns > 32) ns = 32;
        if (ns < 1) ns = 1;
        ctx->nsplit = ns;
        int cap = (int)((S + ns - 1) / ns);
        if (cap < ctx->min_chunk) cap = ctx->min_chunk;
        const int G = NT / (int)(hs / 4);
        ctx->attn_smem = (int)(((uint64_t)G * hs + cap) * sizeof(float));
        if (ctx->attn_smem > kMaxDynSmem) {
            ctx->err = "seq_len too large for the attention kernel's shared memory";
            g_create_error = ctx->err;
            return L2B_ERR_UNSUPPORTED;
        }
        L2B_TRY(cuda_try(ctx, cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem), "cudaFuncSetAttribute"));
        L2B_TRY(dev_alloc(ctx, &ctx->part_o, (size_t)ctx->heads_loc * ns * hs));
        L2B_TRY(dev_alloc(ctx, &ctx->part_ml, (size_t)ctx->heads_loc * ns * 2));
        L2B_TRY(dev_alloc(ctx, &ctx->counters, (size_t)ctx->heads_loc));
        L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->counters, 0, ctx->heads_loc * sizeof(unsigned int), ctx->stream), "memset"));
    }

    // ---- RoPE table (:338-342); the host's own libm values when the caller passes them
    {
        std::vector<float> hc(S * hs / 2), hsn(S * hs / 2);
        if (rope_from) {
            L2B_TRY(cuda_try(ctx, cudaMemcpy(hc.data(), rope_from->rope_cos, hc.size() * sizeof(float), cudaMemcpyDeviceToHost), "rope copy"));
            L2B_TRY(cuda_try(ctx, cudaMemcpy(hsn.data(), rope_from->rope_sin, hsn.size() * sizeof(float), cudaMemcpyDeviceToHost), "rope copy"));
        } else if (rope_cos && rope_sin) {
            memcpy(hc.data(), rope_cos, hc.size() * sizeof(float));
            memcpy(hsn.data(), rope_sin, hsn.size() * sizeof(float));
        } else {
            for (uint64_t p = 0; p < S; ++p)
                for (uint64_t j = 0; j < hs / 2; ++j) {
                    const float head_dim = (float)(2 * j);                                   // i % head_size
                    const float freq = 1.0f / powf(10000.0f, head_dim / (float)hs);          // :339
                    const float val = (float)p * freq;                                       // :340
                    hc[p * (hs / 2) + j] = cosf(val);                                        // :341
                    hsn[p * (hs / 2) + j] = sinf(val);                                       // :342
                }
        }
        L2B_TRY(cuda_try(ctx, cudaMemcpy(ctx->rope_cos, hc.data(), hc.size() * sizeof(float), cudaMemcpyHostToDevice), "rope upload"));
        L2B_TRY(cuda_try(ctx, cudaMemcpy(ctx->rope_sin, hsn.data(), hsn.size() * sizeof(float), cudaMemcpyHostToDevice), "rope upload"));
    }

    // ---- pinned host buffers
    L2B_TRY(cuda_try(ctx, cudaHostAlloc((void **)&ctx->h_logits, V * sizeof(float), cudaHostAllocDefault), "cudaHostAlloc"));
    L2B_TRY(cuda_try(ctx, cudaHostAlloc((void **)&ctx->h_ctl, 2 * CTL_WORDS * sizeof(int), cudaHostAllocDefault), "cudaHostAlloc"));
    L2B_TRY(cuda_try(ctx, cudaHostAlloc((void **)&ctx->h_ints, 16 * sizeof(int), cudaHostAllocDefault), "cudaHostAlloc"));
    L2B_TRY(cuda_try(ctx, cudaHostAlloc((void **)&ctx->h_gen, S * sizeof(int), cudaHostAllocDefault), "cudaHostAlloc"));
    L2B_TRY(cuda_try(ctx, cudaHostAlloc((void **)&ctx->h_cand, (size_t)kCandCap * sizeof(ProbIndex), cudaHostAllocDefault), "cudaHostAlloc"));
    memset(ctx->h_ctl, 0, 2 * CTL_WORDS * sizeof(int));

    // ---- tensor-parallel landing areas: one zeroed arena
    if (world > 1) {
        const size_t slots = 2 * (size_t)L;
        size_t o = 0;
        ctx->off_red = o;    o += slots * world * dim * sizeof(unsigned long long);
        ctx->off_logits = o; o += (size_t)V * sizeof(unsigned long long);
        ctx->off_amax = o;   o += (size_t)world * 2 * sizeof(unsigned long long);
        ctx->arena_bytes = (o + 255) & ~(size_t)255;
        L2B_TRY(dev_alloc(ctx, &ctx->arena, ctx->arena_bytes));
        L2B_TRY(cuda_try(ctx, cudaMemsetAsync(ctx->arena, 0, ctx->arena_bytes, ctx->stream), "memset"));
        ctx->peer_arena[rank] = ctx->arena;
    }

    {
        const char *env = getenv("L2B_NO_GRAPH");
        ctx->use_graphs = !(env && env[0] == '1');
        const char *env2 = getenv("L2B_NO_PDL");
        ctx->use_pdl = !(env2 && env2[0] == '1');
        const char *envts = getenv("L2B_TIME_STEPS");
        ctx->time_steps = envts && envts[0] == '1';
        const char *env3 = getenv("L2B_GEMV8_MIN_BYTES");
        if (env3) ctx->gemv8_min_bytes = atoll(env3);
        const char *env4 = getenv("L2B_GEMV_BIG");
        if (env4 && strcmp(env4, "ldg") == 0) ctx->big_kernel_tma = false;
        const char *env5 = getenv("L2B_TMA_STAGES");
        if (env5) ctx->tma_stages = atoi(env5);
        const char *enva = getenv("L2B_ATTN");
        if (enva && strcmp(enva, "3pass") == 0) ctx->attn_flash = false;
        const char *envpf = getenv("L2B_TMA_PREFILL");
        if (envpf) ctx->tma_prefill = atoi(envpf);
        const char *envs = getenv("L2B_SPIN_TIMEOUT_MS");
        if (envs && atoll(envs) > 0) ctx->spin_ns = (unsigned long long)atoll(envs) * 1000000ull;
        const char *envt = getenv("L2B_TRACE");
        if (envt && envt[0] == '1') {
            ctx->trace_launches = 5 * cfg->n_layers + 4;
            L2B_TRY(dev_alloc(ctx, &ctx->trace, (size_t)ctx->trace_launches * TRACE_MAX_CTAS * TRACE_SLOTS));
            L2B_TRY(cuda_try(ctx, cudaMemset(ctx->trace, 0, (size_t)ctx->trace_launches * TRACE_MAX_CTAS * TRACE_SLOTS * 8), "memset"));
        }
        const char *envn = getenv("L2B_BIG_MIN_N");
        if (envn && atoi(envn) >= 4) ctx->big_min_n = atoi(envn);
        const char *envp = getenv("L2B_TPR_TILES");
        if (envp) ctx->tpr_min_tiles_per_sm = atoi(envp);
        const char *env6 = getenv("L2B_TMA_CTAS");
        if (env6) ctx->tma_ctas_per_sm = atoi(env6) > 0 ? atoi(env6) : 1;
    }
    L2B_TRY(cuda_try(ctx, cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize"));
    return L2B_OK;
}

// ---- creation, stage 2: one eager call of each flavour on every local rank.  It sets function
// attributes outside capture and surfaces launch errors before a graph hides them (it scribbles
// on KV row 0, rewritten by step 0).  Tensor-parallel ranks exchange data during these steps, so
// all local ranks are enqueued before any is synchronised.
int warm_up(const std::vector<l2b_ctx *> &ranks) {
    for (int which = 0; which < G_COUNT; ++which) {
        for (l2b_ctx *ctx : ranks) {
            L2B_TRY(cuda_try(ctx, cudaSetDevice(ctx->device), "cudaSetDevice"));
            memset(ctx->h_ctl, 0, CTL_WORDS * sizeof(int));
            ctx->h_ctl[CTL_TEMP] = 0x3f800000;   // 1.0f
            ctx->h_ctl[CTL_TOPP] = 0x3f666666;   // 0.9f
            if (which == G_ARGMAX_LOOP || which == G_PREFILL_LOOP)
                L2B_TRY(cuda_try(ctx, cudaMemcpyAsync(ctx->ctl, ctx->h_ctl, CTL_HOST_WORDS * sizeof(int), cudaMemcpyHostToDevice, ctx->stream), "ctl upload"));
            L2B_TRY(enqueue_call(ctx, ctx->stream, which));
        }
        for (l2b_ctx *ctx : ranks) {
            L2B_TRY(cuda_try(ctx, cudaSetDevice(ctx->device), "cudaSetDevice"));
            L2B_TRY(cuda_try(ctx, cudaStreamSynchronize(ctx->stream), "warm-up step"));
            L2B_TRY(cuda_try(ctx, cudaGetLastError(), "warm-up step"));
            if (ctx->h_ctl[CTL_WORDS + CTL_ERR] && which != G_ARGMAX_LOOP && which != G_PREFILL_LOOP) {
                ctx->err = "tensor-parallel warm-up step timed out waiting for a peer";
                g_create_error = ctx->err;
                return L2B_ERR_COMM;
            }
        }
    }
    for (l2b_ctx *ctx : ranks) {
        L2B_TRY(cuda_try(ctx, cudaSetDevice(ctx->device), "cudaSetDevice"));
        if (ctx->use_graphs) L2B_TRY(build_graphs(ctx));
    }
    return L2B_OK;
}

// ---- one process per GPU: communicator + CUDA IPC exchange of the arena handles ---------------
int connect_ipc(l2b_ctx *ctx, const l2b_shard *shard) {
    const int world = ctx->world, rank = ctx->rank;
    std::string e;
    if (!nccl_load(&e)) { ctx->err = e; g_create_error = e; return L2B_ERR_COMM; }
    ncclUniqueId id;
    memcpy(&id, shard->comm_id, sizeof id);
    ncclResult_t r = g_nccl.CommInitRank(&ctx->comm, world, id, rank);
    if (r != ncclSuccess) {
        ctx->err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r);
        g_create_error = ctx->err;
        return L2B_ERR_COMM;
    }
    const char *mode = getenv("L2B_TP");
    const bool want = !(mode && strcmp(mode, "nccl") == 0);
    int ok = want ? 1 : 0;
    cudaIpcMemHandle_t hx{};
    if (ok && cudaIpcGetMemHandle(&hx, ctx->arena) != cudaSuccess) {
        cudaGetLastError();
        ok = 0;
    }
    // every rank learns every rank's handle (and whether it could make one) through NCCL
    struct Msg { cudaIpcMemHandle_t hx; int ok; int pad[3]; };
    static_assert(sizeof(Msg) % 16 == 0, "Msg must be 16-byte sized");
    Msg mine{hx, ok, {0, 0, 0}};
    Msg *d_all = nullptr;
    L2B_TRY(dev_alloc(ctx, &d_all, (size_t)world));
    L2B_TRY(cuda_try(ctx, cudaMemcpyAsync(d_all + rank, &mine, sizeof(Msg), cudaMemcpyHostToDevice, ctx->stream), "msg upload"));
    if (g_nccl.AllGather(d_all + rank, d_all, sizeof(Msg), ncclChar, ctx->comm, ctx->stream) != ncclSuccess) {
        ctx->err = "ncclAllGather(ipc handles) failed"; g_create_error = ctx->err; return L2B_ERR_COMM;
    }
    std::vector<Msg> all(world);
    L2B_TRY(cuda_try(ctx, cudaMemcpyAsync(all.data(), d_all, sizeof(Msg) * world, cudaMemcpyDeviceToHost, ctx->stream), "msg download"));
    L2B_TRY(cuda_try(ctx, cudaStreamSynchronize(ctx->stream), "ipc exchange"));
    for (int q = 0; q < world; ++q) ok = ok && all[q].ok;
    if (ok) {
        for (int q = 0; q < world && ok; ++q) {
            if (q == rank) continue;
            void *px = nullptr;
            if (cudaIpcOpenMemHandle(&px, all[q].hx, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                ok = 0;
                break;
            }
            ctx->ipc_opened.push_back(px);
            ctx->peer_arena[q] = (unsigned char *)px;
        }
    }
    // all ranks must take the same path: agree through a max-reduce of the failure bit
    int *d_bad = nullptr;
    L2B_TRY(dev_alloc(ctx, &d_bad, (size_t)1));
    int bad = ok ? 0 : 1;
    L2B_TRY(cuda_try(ctx, cudaMemcpyAsync(d_bad, &bad, sizeof(int), cudaMemcpyHostToDevice, ctx->stream), "flag upload"));
    if (g_nccl.AllReduce(d_bad, d_bad, 1, ncclInt, ncclMax, ctx->comm, ctx->stream) != ncclSuccess) {
        ctx->err = "ncclAllReduce(ipc agreement) failed"; g_create_error = ctx->err; return L2B_ERR_COMM;
    }
    L2B_TRY(cuda_try(ctx, cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream), "flag download"));
    L2B_TRY(cuda_try(ctx, cudaStreamSynchronize(ctx->stream), "ipc agreement"));
    ctx->use_p2p = (bad == 0);
    return L2B_OK;
}

void destroy_rank(l2b_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    // graphs first: NCCL keeps a communicator alive (ncclCommDestroy spins) while captured
    // graphs still reference it
    for (int i = 0; i < G_COUNT; ++i)
        if (ctx->graphs[i]) cudaGraphExecDestroy(ctx->graphs[i]);
    cudaDeviceSynchronize();
    if (ctx->comm && g_nccl.ok) g_nccl.CommDestroy(ctx->comm);
    for (void *p : ctx->ipc_opened) cudaIpcCloseMemHandle(p);
    for (void *p : ctx->owned) cudaFree(p);
    for (int i = 0; i < 2; ++i) {
        if (ctx->stage[i]) cudaFreeHost(ctx->stage[i]);
        if (ctx->stage_ev[i]) cudaEventDestroy(ctx->stage_ev[i]);
    }
    if (ctx->h_logits) cudaFreeHost(ctx->h_logits);
    if (ctx->h_ctl) cudaFreeHost(ctx->h_ctl);
    if (ctx->h_ints) cudaFreeHost(ctx->h_ints);
    if (ctx->h_gen) cudaFreeHost(ctx->h_gen);
    if (ctx->h_cand) cudaFreeHost(ctx->h_cand);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

void destroy_all(l2b_ctx *ctx) {
    if (!ctx) return;
    std::vector<l2b_ctx *> ranks = locals(ctx);
    // every rank must be idle before any rank's memory (a peer's landing area) goes away
    for (l2b_ctx *c : ranks) { cudaSetDevice(c->device); if (c->stream) cudaStreamSynchronize(c->stream); }
    for (size_t i = ranks.size(); i-- > 0;) destroy_rank(ranks[i]);
}

int common_create(l2b_ctx **out, const l2b_config *cfg, const Source &src, uint64_t n_floats,
                  const float *rope_cos, const float *rope_sin, const l2b_shard *shard, int n_gpus) {
    if (!out || !cfg) { g_create_error = "NULL argument"; return L2B_ERR_INVALID_ARG; }
    *out = nullptr;
    const bool in_process = n_gpus > 1;
    const int world = shard ? shard->world_size : n_gpus;
    std::string why;
    int rc = validate_config(cfg, world, &why);
    if (rc) { g_create_error = why; return rc; }
    if (shard && (shard->rank < 0 || shard->rank >= world)) { g_create_error = "rank out of range"; return L2B_ERR_INVALID_ARG; }
    if (src.host && n_floats < checkpoint_floats(cfg)) {
        g_create_error = "host_weights shorter than the checkpoint layout requires";
        return L2B_ERR_INVALID_ARG;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        g_create_error = "no CUDA device";
        return L2B_ERR_NO_DEVICE;
    }
    if (in_process && ndev < n_gpus) { g_create_error = "fewer CUDA devices than n_gpus"; return L2B_ERR_NO_DEVICE; }
    const int device0 = shard ? shard->device : 0;
    if (device0 < 0 || device0 >= ndev) { g_create_error = "device ordinal out of range"; return L2B_ERR_INVALID_ARG; }

    std::vector<l2b_ctx *> ranks;
    auto bail = [&](int code) {
        for (size_t i = ranks.size(); i-- > 0;) destroy_rank(ranks[i]);
        return code;
    };
    const int nlocal = in_process ? n_gpus : 1;
    for (int i = 0; i < nlocal; ++i) {
        l2b_ctx *ctx = new l2b_ctx();
        ranks.push_back(ctx);
        const int rank = in_process ? i : (shard ? shard->rank : 0);
        const int device = in_process ? i : device0;
        rc = create_rank(ctx, cfg, src, rope_cos, rope_sin, rank, world, device);
        if (rc) return bail(rc);
    }
    if (in_process) {
        // one process drives all GPUs: peers are plain UVA pointers once peer access is on
        for (l2b_ctx *a : ranks) {
            cudaSetDevice(a->device);
            for (l2b_ctx *b : ranks) {
                if (a == b) continue;
                int can = 0;
                cudaDeviceCanAccessPeer(&can, a->device, b->device);
                if (!can) { g_create_error = "GPUs are not peer-accessible (NVLink/NVSwitch required for n_gpus > 1)"; return bail(L2B_ERR_COMM); }
                cudaError_t e = cudaDeviceEnablePeerAccess(b->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { g_create_error = std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e); return bail(L2B_ERR_COMM); }
                cudaGetLastError();
                a->peer_arena[b->rank] = b->arena;
            }
            a->use_p2p = true;
            a->leader = ranks[0];
        }
    } else if (world > 1) {
        rc = connect_ipc(ranks[0], shard);
        if (rc) return bail(rc);
    }
    rc = warm_up(ranks);
    if (rc) return bail(rc);
    if (in_process) ranks[0]->members = ranks;
    *out = ranks[0];
    return L2B_OK;
}
#undef L2B_TRY

// ---- running a call on every local rank -------------------------------------------------------
void fill_ctl(l2b_ctx *ctx, int token, int pos, int stop_on_bos, float temperature, float top_p) {
    int *h = ctx->h_ctl;
    h[CTL_TOKEN] = token; h[CTL_POS] = pos; h[CTL_DONE] = 0; h[CTL_STEP] = 0;
    h[CTL_STOP_ON_BOS] = stop_on_bos;
    memcpy(&h[CTL_TEMP], &temperature, sizeof(float));
    memcpy(&h[CTL_TOPP], &top_p, sizeof(float));
}

int finish_call(l2b_ctx *lead, const std::vector<l2b_ctx *> &ranks) {
    int rc = L2B_OK;
    for (l2b_ctx *c : ranks) {
        cudaSetDevice(c->device);
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess && rc == L2B_OK) {
            lead->err = std::string("step failed: ") + cudaGetErrorString(e);
            rc = L2B_ERR_CUDA;
        }
        if (c->h_ctl[CTL_WORDS + CTL_ERR] && rc == L2B_OK) {
            lead->err = "tensor-parallel exchange timed out: a peer rank died or fell out of lockstep";
            rc = L2B_ERR_COMM;
        }
    }
    return rc;
}

// run one step; which: G_LOGITS / G_ARGMAX_ONE / G_SAMPLE
int run_step(l2b_ctx *lead, int token, int pos, int which, float temperature, float top_p) {
    // One step costs a small model ~90 us on the device, so every host call here is on the clock of
    // the end-to-end loop: no per-step events unless asked for (L2B_TIME_STEPS=1), no allocation.
    l2b_ctx *single[1] = {lead};
    l2b_ctx *const *ranks = lead->members.empty() ? single : lead->members.data();
    const size_t nranks = lead->members.empty() ? 1 : lead->members.size();
    for (size_t i = 0; i < nranks; ++i) {
        l2b_ctx *ctx = ranks[i];
        if (nranks > 1 || i == 0) L2B_CUDA(lead, cudaSetDevice(ctx->device));
        fill_ctl(ctx, token, pos, 0, temperature, top_p);
        ctx->last_launches = 0;
        if (ctx == lead && lead->time_steps) L2B_CUDA(lead, cudaEventRecord(ctx->ev0, ctx->stream));
        if (ctx->use_graphs) {
            L2B_CUDA(lead, cudaGraphLaunch(ctx->graphs[which], ctx->stream));
            ctx->last_launches = ctx->launches_per_step + (which == G_LOGITS ? 0 : 1);
        } else {
            int rc = enqueue_call(ctx, ctx->stream, which);
            if (rc) { lead->err = ctx->err; return rc; }
        }
        if (ctx == lead && lead->time_steps) L2B_CUDA(lead, cudaEventRecord(ctx->ev1, ctx->stream));
    }
    int rc = L2B_OK;
    for (size_t i = 0; i < nranks; ++i) {
        l2b_ctx *c = ranks[i];
        if (nranks > 1) cudaSetDevice(c->device);
        cudaError_t e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess && rc == L2B_OK) {
            lead->err = std::string("step failed: ") + cudaGetErrorString(e);
            rc = L2B_ERR_CUDA;
        }
        if (c->h_ctl[CTL_WORDS + CTL_ERR] && rc == L2B_OK) {
            lead->err = "tensor-parallel exchange timed out: a peer rank died or fell out of lockstep";
            rc = L2B_ERR_COMM;
        }
    }
    if (rc) return rc;
    if (lead->time_steps) {
        if (nranks > 1) L2B_CUDA(lead, cudaSetDevice(lead->device));
        L2B_CUDA(lead, cudaEventElapsedTime(&lead->last_ms, lead->ev0, lead->ev1));
    }
    if (pos + 1 > lead->n_appended) lead->n_appended = pos + 1;
    return L2B_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------
extern "C" {

int32_t l2b_abi_version(void) { return L2B_ABI_VERSION; }

const char *l2b_status_string(int32_t s) {
    switch (s) {
    case L2B_OK: return "ok";
    case L2B_ERR_INVALID_ARG: return "invalid argument";
    case L2B_ERR_UNSUPPORTED: return "unsupported shape";
    case L2B_ERR_CUDA: return "CUDA error";
    case L2B_ERR_NO_DEVICE: return "no usable sm_100 device";
    case L2B_ERR_OOM: return "out of memory";
    case L2B_ERR_COMM: return "communication error";
    case L2B_ERR_STATE: return "call order violated";
    default: return "unknown status";
    }
}

const char *l2b_last_error(const l2b_ctx *ctx) {
    if (!ctx) return g_create_error.c_str();
    return ctx->err.empty() ? kNoError : ctx->err.c_str();
}

uint64_t l2b_checkpoint_floats(const l2b_config *cfg) { return cfg ? checkpoint_floats(cfg) : 0; }

int32_t l2b_create(l2b_ctx **out, const l2b_config *cfg, const float *host_weights, uint64_t n_floats,
                   const float *rope_cos, const float *rope_sin, int32_t n_gpus) {
    if (!host_weights) { g_create_error = "host_weights is NULL"; return L2B_ERR_INVALID_ARG; }
    if (n_gpus != 1 && n_gpus != 2 && n_gpus != 4 && n_gpus != 8) {
        g_create_error = "n_gpus must be 1, 2, 4 or 8";
        return L2B_ERR_UNSUPPORTED;
    }
    Source s; s.host = host_weights;
    return common_create(out, cfg, s, n_floats, rope_cos, rope_sin, nullptr, n_gpus);
}

int32_t l2b_create_sharded(l2b_ctx **out, const l2b_config *cfg, const float *host_weights,
                           uint64_t n_floats, const float *rope_cos, const float *rope_sin,
                           const l2b_shard *shard) {
    if (!host_weights || !shard) { g_create_error = "NULL argument"; return L2B_ERR_INVALID_ARG; }
    Source s; s.host = host_weights;
    return common_create(out, cfg, s, n_floats, rope_cos, rope_sin, shard, 1);
}

int32_t l2b_create_synthetic(l2b_ctx **out, const l2b_config *cfg, uint64_t seed, const l2b_shard *shard) {
    Source s; s.host = nullptr; s.seed = seed;
    return common_create(out, cfg, s, 0, nullptr, nullptr, shard, 1);
}

int32_t l2b_create_synthetic_group(l2b_ctx **out, const l2b_config *cfg, uint64_t seed, int32_t n_gpus) {
    if (n_gpus != 1 && n_gpus != 2 && n_gpus != 4 && n_gpus != 8) {
        g_create_error = "n_gpus must be 1, 2, 4 or 8";
        return L2B_ERR_UNSUPPORTED;
    }
    Source s; s.host = nullptr; s.seed = seed;
    return common_create(out, cfg, s, 0, nullptr, nullptr, nullptr, n_gpus);
}

void l2b_destroy(l2b_ctx *ctx) { destroy_all(ctx); }

int32_t l2b_reset(l2b_ctx *ctx) {
    if (!ctx) return L2B_ERR_INVALID_ARG;
    ctx->n_appended = 0;
    return L2B_OK;
}

float *l2b_logits_buffer(l2b_ctx *ctx) { return ctx ? ctx->h_logits : nullptr; }

int32_t l2b_forward_pinned(l2b_ctx *ctx, int32_t token, int32_t pos, const float **logits) {
    int rc = check_step_args(ctx, token, pos);
    if (rc) return rc;
    if (!logits) return fail(ctx, L2B_ERR_INVALID_ARG, "logits is NULL");
    rc = run_step(ctx, token, pos, G_LOGITS, 1.0f, 0.0f);
    if (rc) return rc;
    *logits = ctx->h_logits;
    return L2B_OK;
}

int32_t l2b_forward(l2b_ctx *ctx, int32_t token, int32_t pos, float *host_logits) {
    int rc = check_step_args(ctx, token, pos);
    if (rc) return rc;
    if (!host_logits) return fail(ctx, L2B_ERR_INVALID_ARG, "host_logits is NULL");
    rc = run_step(ctx, token, pos, G_LOGITS, 1.0f, 0.0f);
    if (rc) return rc;
    // state.logits of the reference is one long-lived buffer (src/main.zig:149).  A host that
    // adopted l2b_logits_buffer() as that buffer gets the logits without a second copy; any other
    // destination gets one streaming memcpy from the pinned landing buffer.
    if (host_logits != ctx->h_logits)
        memcpy(host_logits, ctx->h_logits, (size_t)ctx->cfg.vocab_size * sizeof(float));
    return L2B_OK;
}

int32_t l2b_forward_argmax(l2b_ctx *ctx, int32_t token, int32_t pos, int32_t *next) {
    int rc = check_step_args(ctx, token, pos);
    if (rc) return rc;
    if (!next) return fail(ctx, L2B_ERR_INVALID_ARG, "next is NULL");
    rc = run_step(ctx, token, pos, G_ARGMAX_ONE, 1.0f, 0.0f);
    if (rc) return rc;
    *next = ctx->h_ints[0];
    return L2B_OK;
}

int32_t l2b_forward_sample(l2b_ctx *ctx, int32_t token, int32_t pos, float temperature, float top_p,
                           float *host_probs, l2b_prob_index *cand, int32_t cand_cap, int32_t *n_cand) {
    int rc = check_step_args(ctx, token, pos);
    if (rc) return rc;
    if (!(temperature > 0.0f)) return fail(ctx, L2B_ERR_INVALID_ARG, "temperature must be > 0 (use l2b_forward_argmax for 0)");
    if (top_p < 0.0f || top_p > 1.0f) return fail(ctx, L2B_ERR_INVALID_ARG, "top_p must be in [0, 1]");
    const bool filter = (top_p != 0.0f && top_p != 1.0f);            // :1009
    if (filter && (!cand || !n_cand || cand_cap <= 0)) return fail(ctx, L2B_ERR_INVALID_ARG, "candidate buffer missing");
    rc = run_step(ctx, token, pos, G_SAMPLE, temperature, filter ? top_p : -1.0f);
    if (rc) return rc;
    const int V = ctx->cfg.vocab_size;
    if (host_probs && host_probs != ctx->h_logits) memcpy(host_probs, ctx->h_logits, (size_t)V * sizeof(float));
    if (n_cand) *n_cand = 0;
    if (filter) {
        const int n = ctx->h_ints[2];
        if (n > kCandCap || n > cand_cap) { *n_cand = -n; return L2B_OK; }   // too many: filter host_probs on the host
        static_assert(sizeof(l2b_prob_index) == sizeof(ProbIndex), "candidate layout");
        memcpy(cand, ctx->h_cand, (size_t)n * sizeof(ProbIndex));
        *n_cand = n;
    }
    return L2B_OK;
}

}  // extern "C" (templates below)

// ---- batched passes over the weights (csrc/l2b_prefill.cuh) ------------------------------------
typedef void (*pf_fn)(const PrefillParams);
template <int NB>
pf_fn pf_pick(int epi) {
    switch (epi) {
    case EPI_QKV: return prefill_gemm_kernel<EPI_QKV, NB>;
    case EPI_SILU: return prefill_gemm_kernel<EPI_SILU, NB>;
    case EPI_STORE: return prefill_gemm_kernel<EPI_STORE, NB>;
    case EPI_ARGMAX: return prefill_gemm_kernel<EPI_ARGMAX, NB>;
    default: return prefill_gemm_kernel<EPI_RESID, NB>;
    }
}
constexpr size_t kPfSmemBudget = 227 * 1024 - 8192;   // the prefill kernels keep ~6.5 KB of static shared memory

// scratch of the batched passes, once per set of weights (every context over them uses it in turn)
static int alloc_batch_scratch(l2b_ctx *ctx, WeightStore &w) {
    const size_t B = L2B_MAX_BATCH, S = ctx->cfg.seq_len, V = ctx->cfg.vocab_size;
    const size_t nvec = S > B ? S : B;
    int rc;
    if ((rc = dev_alloc(ctx, &w.x, B * ctx->dim))) return rc;
    if ((rc = dev_alloc(ctx, &w.q, B * ctx->q_loc))) return rc;
    if ((rc = dev_alloc(ctx, &w.xb, B * ctx->q_loc))) return rc;
    if ((rc = dev_alloc(ctx, &w.hb, B * ctx->hid_loc))) return rc;
    if ((rc = dev_alloc(ctx, &w.logits, B * V))) return rc;
    if ((rc = dev_alloc(ctx, &w.part_o, B * ctx->heads_loc * ctx->nsplit * ctx->head_size))) return rc;
    if ((rc = dev_alloc(ctx, &w.part_ml, B * ctx->heads_loc * ctx->nsplit * 2))) return rc;
    if ((rc = dev_alloc(ctx, &w.counters, B * ctx->heads_loc))) return rc;
    if ((rc = dev_alloc(ctx, &w.amax, B))) return rc;
    if ((rc = dev_alloc(ctx, &w.vec, nvec))) return rc;
    if ((rc = dev_alloc(ctx, &w.forced, B * S))) return rc;
    if ((rc = dev_alloc(ctx, &w.out, B * S))) return rc;
    if ((rc = dev_alloc(ctx, &w.n_done, B))) return rc;
    L2B_CUDA(ctx, cudaMemsetAsync(w.counters, 0, B * ctx->heads_loc * sizeof(unsigned int), ctx->stream));
    void *h = nullptr;
    L2B_CUDA(ctx, cudaHostAlloc(&h, nvec * sizeof(BatchVec), cudaHostAllocDefault));
    w.pinned.push_back(h); w.h_vec = static_cast<BatchVec *>(h);
    L2B_CUDA(ctx, cudaHostAlloc(&h, B * V * sizeof(float), cudaHostAllocDefault));
    w.pinned.push_back(h); w.h_logits = static_cast<float *>(h);
    L2B_CUDA(ctx, cudaHostAlloc(&h, (B * S + B) * sizeof(int), cudaHostAllocDefault));
    w.pinned.push_back(h); w.h_ints = static_cast<int *>(h);
    L2B_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return L2B_OK;
}

// can this context run PF_MAXB vectors per weight pass?  Single GPU, flash attention, and all four
// per-layer GEMVs bandwidth-bound shapes of the TMA-ring kernel; otherwise l2b_prefill runs the
// positions one by one on the device and the batch calls run each stream's own step in turn (same
// results, weights streamed once per token).
static int pf_prepare(l2b_ctx *ctx) {
    if (ctx->pf_ready) return L2B_OK;
    ctx->pf_ready = true;
    const char *env = getenv("L2B_PREFILL_BATCH");
    if (env && env[0] == '0') return L2B_OK;
    const uint64_t dim = ctx->dim, hid = ctx->hid_loc;
    size_t smem = 0;
    const bool shapes_ok = ctx->world == 1 && !ctx->leader && dim >= (uint64_t)ctx->big_min_n && hid >= (uint64_t)ctx->big_min_n &&
                           dim <= 5 * (TMA_THREADS - 32) * 4 && ctx->gemv8_min_bytes >= 0 &&
                           dim * dim * 4 >= (uint64_t)ctx->gemv8_min_bytes && ctx->attn_flash &&
                           pick_attention(ctx->head_size, true, &smem) != attention_kernel &&
                           (kPfSmemBudget - PF_MAXB * dim * 4) / ((size_t)TMA_STAGE_FLOATS * 4) >= 2 &&
                           (kPfSmemBudget - 2 * hid * 4) / ((size_t)TMA_STAGE_FLOATS * 4) >= 2;
    if (!shapes_ok) return L2B_OK;
    L2B_CUDA(ctx, cudaSetDevice(ctx->device));
    WeightStore &w = *ctx->weights;
    if (!w.batch_ready) {
        const size_t mark = ctx->owned.size();
        const int rc = alloc_batch_scratch(ctx, w);
        w.owned.insert(w.owned.end(), ctx->owned.begin() + mark, ctx->owned.end());   // the store frees them
        ctx->owned.resize(mark);
        if (rc) return rc;
        w.batch_ready = true;
    }
    for (int epi : {(int)EPI_QKV, (int)EPI_SILU, (int)EPI_RESID, (int)EPI_STORE, (int)EPI_ARGMAX}) {
        L2B_CUDA(ctx, cudaFuncSetAttribute(pf_pick<PF_MAXB>(epi), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPfSmemBudget));
        L2B_CUDA(ctx, cudaFuncSetAttribute(pf_pick<2>(epi), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPfSmemBudget));
    }
    ctx->pf_ok = true;
    return L2B_OK;
}

template <int NB>
static int pf_launch(l2b_ctx *ctx, int epi, PrefillParams p, cudaStream_t st) {
    const size_t xbytes = (size_t)NB * p.n * 4;
    int nstage = (int)((kPfSmemBudget - xbytes) / ((size_t)TMA_STAGE_FLOATS * 4));
    if (nstage > TMA_MAX_STAGES) nstage = TMA_MAX_STAGES;
    p.nstage = nstage;
    int grid = ctx->num_sms;
    const int npairs = (p.total_rows + 1) / 2;
    if (grid > npairs) grid = npairs;
    cudaLaunchConfig_t lc{};
    lc.gridDim = dim3(grid);
    lc.blockDim = dim3(TMA_THREADS);
    lc.dynamicSmemBytes = (size_t)nstage * TMA_STAGE_FLOATS * 4 + xbytes;
    lc.stream = st;
    cudaLaunchAttribute at[1] = {pdl_attr()};
    lc.attrs = at;
    lc.numAttrs = ctx->use_pdl ? 1 : 0;
    L2B_CUDA(ctx, cudaLaunchKernelEx(&lc, pf_pick<NB>(epi), p));
    ++ctx->last_launches;
    return L2B_OK;
}

// Layer l (src/main.zig:305-422) for the n <= L2B_MAX_BATCH vectors vec[0..n) whose residual streams are
// weights->x[0..n): PF_MAXB vectors per pass over the dim-wide weights, two per pass over w2 (its
// hidden-wide inputs fill shared memory), one attention launch for all n.  Prompt prefill and batched
// decode both run their layers through here.
static int enqueue_batch_layer(l2b_ctx *ctx, cudaStream_t st, int l, const BatchVec *vec, int n) {
    const l2b_config &c = ctx->cfg;
    const WeightStore &w = *ctx->weights;
    const int dim = ctx->dim;
    const size_t loff = (size_t)l * c.seq_len * ctx->kv_loc;
    int rc;
    // ---- rmsnorm + q,k,v + RoPE + KV append (:305-358)
    for (int g = 0; g < n; g += PF_MAXB) {
        PrefillParams p{};
        p.n = dim; p.nb = n - g < PF_MAXB ? n - g : PF_MAXB; p.vec = vec + g;
        p.x_in = w.x + (size_t)g * dim;
        if (l == 0) { p.emb = ctx->emb; p.x_out = w.x + (size_t)g * dim; }   // :295-296
        p.gamma = ctx->rms_att + (size_t)l * dim;
        p.w0 = ctx->wq + (size_t)l * ctx->q_loc * dim;
        p.w1 = ctx->wk + (size_t)l * ctx->kv_loc * dim;
        p.w2 = ctx->wv + (size_t)l * ctx->kv_loc * dim;
        p.rows0 = ctx->q_loc; p.rows1 = ctx->kv_loc; p.rows2 = ctx->kv_loc;
        p.total_rows = ctx->q_loc + 2 * ctx->kv_loc;
        p.out0 = w.q + (size_t)g * ctx->q_loc;
        p.kv_off = loff;
        p.rope_cos = ctx->rope_cos; p.rope_sin = ctx->rope_sin;
        p.head_size = ctx->head_size; p.kv_dim = ctx->kv_loc;
        if ((rc = pf_launch<PF_MAXB>(ctx, EPI_QKV, p, st))) return rc;
    }
    // ---- attention of the n queries (:361-389); query z sees positions 0 .. vec[z].pos of its own cache
    {
        size_t attn_smem = 0;
        attn_fn afn = pick_attention(ctx->head_size, true, &attn_smem);
        AttnParams a{};
        a.ctl = ctx->ctl; a.q = w.q; a.vec = vec; a.kv_off = loff;
        a.xb = w.xb; a.part_o = w.part_o; a.part_ml = w.part_ml; a.counters = w.counters;
        a.head_size = ctx->head_size; a.kv_dim = ctx->kv_loc; a.kv_mul = ctx->kv_mul;
        a.nsplit = ctx->nsplit; a.min_chunk = ctx->min_chunk;
        a.q_stride = ctx->q_loc; a.seq_len = c.seq_len;
        cudaLaunchConfig_t lc{};
        lc.gridDim = dim3(ctx->heads_loc, ctx->nsplit, n);
        lc.blockDim = dim3(NT);
        lc.dynamicSmemBytes = attn_smem;
        lc.stream = st;
        cudaLaunchAttribute at[1] = {pdl_attr()};
        lc.attrs = at;
        lc.numAttrs = ctx->use_pdl ? 1 : 0;
        L2B_CUDA(ctx, cudaLaunchKernelEx(&lc, afn, a));
        ++ctx->last_launches;
    }
    // ---- wo + residual (:392-395)
    for (int g = 0; g < n; g += PF_MAXB) {
        PrefillParams o{};
        o.n = ctx->q_loc; o.nb = n - g < PF_MAXB ? n - g : PF_MAXB; o.vec = vec + g;
        o.x_in = w.xb + (size_t)g * ctx->q_loc;
        o.w0 = ctx->wo + (size_t)l * dim * ctx->q_loc;
        o.total_rows = dim; o.rows0 = dim;
        o.out0 = w.x + (size_t)g * dim;
        if ((rc = pf_launch<PF_MAXB>(ctx, EPI_RESID, o, st))) return rc;
    }
    // ---- rmsnorm + w1,w3 + SiLU*mul (:398-416)
    for (int g = 0; g < n; g += PF_MAXB) {
        PrefillParams f{};
        f.n = dim; f.nb = n - g < PF_MAXB ? n - g : PF_MAXB; f.vec = vec + g;
        f.x_in = w.x + (size_t)g * dim;
        f.gamma = ctx->rms_ffn + (size_t)l * dim;
        f.w0 = ctx->w1 + (size_t)l * ctx->hid_loc * dim;
        f.w1 = ctx->w3 + (size_t)l * ctx->hid_loc * dim;
        f.rows0 = ctx->hid_loc;
        f.total_rows = 2 * ctx->hid_loc;
        f.out0 = w.hb + (size_t)g * ctx->hid_loc;
        if ((rc = pf_launch<PF_MAXB>(ctx, EPI_SILU, f, st))) return rc;
    }
    // ---- w2 + residual (:419-422); hidden-sized inputs: two vectors per pass (shared memory)
    for (int b = 0; b < n; b += 2) {
        PrefillParams d{};
        d.n = ctx->hid_loc; d.nb = n - b < 2 ? n - b : 2; d.vec = vec + b;
        d.x_in = w.hb + (size_t)b * ctx->hid_loc;
        d.w0 = ctx->w2 + (size_t)l * dim * ctx->hid_loc;
        d.total_rows = dim; d.rows0 = dim;
        d.out0 = w.x + (size_t)b * dim;
        if ((rc = pf_launch<2>(ctx, EPI_RESID, d, st))) return rc;
    }
    return L2B_OK;
}

// final rmsnorm + classifier (:426-429) of the n vectors: logits rows weights->logits[0..n), and with
// argmax the packed first-maximum key of vector b at weights->amax[b]
static int enqueue_batch_classifier(l2b_ctx *ctx, cudaStream_t st, const BatchVec *vec, int n, bool argmax) {
    const WeightStore &w = *ctx->weights;
    for (int g = 0; g < n; g += PF_MAXB) {
        PrefillParams k{};
        k.n = ctx->dim; k.nb = n - g < PF_MAXB ? n - g : PF_MAXB; k.vec = vec + g;
        k.x_in = w.x + (size_t)g * ctx->dim;
        k.gamma = ctx->rms_final;
        k.w0 = ctx->wcls;
        k.total_rows = ctx->vocab_loc; k.rows0 = ctx->vocab_loc;
        k.out0 = w.logits + (size_t)g * ctx->vocab_loc;
        k.amax = w.amax + g;
        const int rc = pf_launch<PF_MAXB>(ctx, argmax ? EPI_ARGMAX : EPI_STORE, k, st);
        if (rc) return rc;
    }
    return L2B_OK;
}

// n_tokens positions starting at pos0, PF_MAXB per pass over the weights; KV cache filled, no logits
static int prefill_batched(l2b_ctx *ctx, const int32_t *tokens, int n_tokens, int pos0) {
    const l2b_config &c = ctx->cfg;
    WeightStore &w = *ctx->weights;
    cudaStream_t st = ctx->stream;
    L2B_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int i = 0; i < n_tokens; ++i) w.h_vec[i] = BatchVec{tokens[i], pos0 + i, 0, 0, 1, 0, ctx->kcache, ctx->vcache};
    L2B_CUDA(ctx, cudaMemcpyAsync(w.vec, w.h_vec, (size_t)n_tokens * sizeof(BatchVec), cudaMemcpyHostToDevice, st));
    L2B_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
    ctx->last_launches = 0;
    for (int done = 0; done < n_tokens; done += PF_MAXB) {
        const int nb = n_tokens - done < PF_MAXB ? n_tokens - done : PF_MAXB;
        for (int l = 0; l < c.n_layers; ++l) {
            const int rc = enqueue_batch_layer(ctx, st, l, w.vec + done, nb);
            if (rc) return rc;
        }
    }
    L2B_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
    L2B_CUDA(ctx, cudaStreamSynchronize(st));
    L2B_CUDA(ctx, cudaGetLastError());
    L2B_CUDA(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
    if (pos0 + n_tokens > ctx->n_appended) ctx->n_appended = pos0 + n_tokens;
    return L2B_OK;
}

// Decode steps of n streams over one set of weights, every pass over the weights shared by up to
// PF_MAXB of them, on streams[0]'s CUDA stream.  host_logits != nullptr: one step, logits [n][vocab]
// returned.  Otherwise the temperature-0 loop of l2b_generate_argmax for every stream at once: stream k
// takes min(n_steps, seq_len - pos[k]) steps, its tokens chosen by advance_batch_kernel on the device.
static int run_batch(l2b_ctx *const *streams, int n, const int32_t *tokens, const int32_t *pos, int n_steps,
                     const int32_t *forced, int stop_on_bos, float *host_logits, int32_t *out_next, int32_t *n_done) {
    l2b_ctx *lead = streams[0];
    WeightStore &w = *lead->weights;
    cudaStream_t st = lead->stream;
    const size_t S = lead->cfg.seq_len, V = lead->cfg.vocab_size, B = L2B_MAX_BATCH;
    const bool gen = host_logits == nullptr;
    int max_steps = 0;
    for (int k = 0; k < n; ++k) {
        const int room = (int)S - pos[k];
        const int lim = gen ? (n_steps < room ? n_steps : room) : 1;
        w.h_vec[k] = BatchVec{tokens[k], pos[k], lim > 0 ? 0 : 1, 0, lim, 0, streams[k]->kcache, streams[k]->vcache};
        if (lim > max_steps) max_steps = lim;
        for (int i = 0; gen && i < lim; ++i) w.h_ints[k * S + i] = forced ? forced[(size_t)k * n_steps + i] : -1;
    }
    if (max_steps == 0) {
        for (int k = 0; k < n; ++k) n_done[k] = 0;
        return L2B_OK;
    }
    L2B_CUDA(lead, cudaSetDevice(lead->device));
    L2B_CUDA(lead, cudaMemcpyAsync(w.vec, w.h_vec, (size_t)n * sizeof(BatchVec), cudaMemcpyHostToDevice, st));
    if (gen) {
        L2B_CUDA(lead, cudaMemcpyAsync(w.forced, w.h_ints, (size_t)n * S * sizeof(int), cudaMemcpyHostToDevice, st));
        L2B_CUDA(lead, cudaMemsetAsync(w.n_done, 0, (size_t)n * sizeof(int), st));
        L2B_CUDA(lead, cudaMemsetAsync(w.amax, 0, (size_t)n * sizeof(unsigned long long), st));
    }
    L2B_CUDA(lead, cudaEventRecord(lead->ev0, st));
    lead->last_launches = 0;
    int rc;
    for (int i = 0; i < max_steps; ++i) {
        for (int l = 0; l < lead->cfg.n_layers; ++l)
            if ((rc = enqueue_batch_layer(lead, st, l, w.vec, n))) return rc;
        if ((rc = enqueue_batch_classifier(lead, st, w.vec, n, gen))) return rc;
        if (gen) {
            BatchVec *vec = w.vec;
            unsigned long long *amax = w.amax;
            const int *fp = w.forced;
            int *op = w.out, *dp = w.n_done, stride = (int)S, sob = stop_on_bos ? 1 : 0;
            void *args[] = {&vec, &n, &amax, &fp, &op, &dp, &stride, &sob};
            if ((rc = launch_small(lead, (const void *)advance_batch_kernel, dim3(1), dim3(32), args, st, true))) return rc;
        }
    }
    if (gen) {
        L2B_CUDA(lead, cudaMemcpyAsync(w.h_ints, w.out, (size_t)n * S * sizeof(int), cudaMemcpyDeviceToHost, st));
        L2B_CUDA(lead, cudaMemcpyAsync(w.h_ints + B * S, w.n_done, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
    } else {
        L2B_CUDA(lead, cudaMemcpyAsync(w.h_logits, w.logits, (size_t)n * V * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    L2B_CUDA(lead, cudaEventRecord(lead->ev1, st));
    L2B_CUDA(lead, cudaStreamSynchronize(st));
    L2B_CUDA(lead, cudaGetLastError());
    L2B_CUDA(lead, cudaEventElapsedTime(&lead->last_ms, lead->ev0, lead->ev1));
    for (int k = 0; k < n; ++k) {
        const int steps = gen ? w.h_ints[B * S + k] : 1;
        if (gen) {
            n_done[k] = steps;
            for (int i = 0; i < steps; ++i) out_next[(size_t)k * n_steps + i] = w.h_ints[k * S + i];
        }
        if (pos[k] + steps > streams[k]->n_appended) streams[k]->n_appended = pos[k] + steps;
    }
    if (!gen) memcpy(host_logits, w.h_logits, (size_t)n * V * sizeof(float));
    return L2B_OK;
}

// argument checks of the batch calls (before any CUDA call); errors land on streams[0] when there is one
static int check_batch_args(l2b_ctx *const *streams, int n, const int32_t *tokens, const int32_t *pos) {
    if (!streams || !tokens || !pos) { g_create_error = "NULL argument"; return L2B_ERR_INVALID_ARG; }
    if (n < 1 || n > L2B_MAX_BATCH) {
        g_create_error = "n must be 1 .. L2B_MAX_BATCH";
        return fail(n > 0 ? streams[0] : nullptr, L2B_ERR_INVALID_ARG, "n must be 1 .. L2B_MAX_BATCH");
    }
    for (int k = 0; k < n; ++k)
        if (!streams[k]) { g_create_error = "NULL stream"; return fail(streams[0], L2B_ERR_INVALID_ARG, "NULL stream"); }
    for (int k = 0; k < n; ++k) {
        for (int j = 0; j < k; ++j)
            if (streams[j] == streams[k]) return fail(streams[0], L2B_ERR_INVALID_ARG, "the same stream is listed twice");
        if (!streams[k]->weights || streams[k]->weights != streams[0]->weights)
            return fail(streams[0], L2B_ERR_INVALID_ARG, "streams over different weights");
    }
    for (int k = 0; k < n; ++k) {
        const int rc = check_step_args(streams[k], tokens[k], pos[k]);
        if (rc) {
            if (k) streams[0]->err = "stream " + std::to_string(k) + ": " + streams[k]->err;
            return rc;
        }
    }
    return L2B_OK;
}

extern "C" {

// n_steps replays of a device-loop graph (G_ARGMAX_LOOP or G_PREFILL_LOOP) starting at (token, pos)
static int run_device_loop(l2b_ctx *ctx, int which, int token, int pos, int n_steps, const int32_t *forced,
                           int stop_on_bos, int *done_out) {
    std::vector<l2b_ctx *> ranks = locals(ctx);
    int launches = 0, rc;
    for (l2b_ctx *c : ranks) {
        L2B_CUDA(ctx, cudaSetDevice(c->device));
        // forced tokens (prompt forcing, :999-1000); -1 = free-running
        for (int i = 0; i < n_steps; ++i) c->h_gen[i] = forced ? forced[i] : -1;
        L2B_CUDA(ctx, cudaMemcpyAsync(c->gen_forced, c->h_gen, (size_t)n_steps * sizeof(int),
                                      cudaMemcpyHostToDevice, c->stream));
        L2B_CUDA(ctx, cudaMemsetAsync(c->gen_ndone, 0, sizeof(int), c->stream));
        L2B_CUDA(ctx, cudaMemsetAsync(c->amax, 0, sizeof(unsigned long long), c->stream));
        fill_ctl(c, token, pos, stop_on_bos ? 1 : 0, 1.0f, -1.0f);
        if (c == ctx) L2B_CUDA(ctx, cudaEventRecord(c->ev0, c->stream));
        L2B_CUDA(ctx, cudaMemcpyAsync(c->ctl, c->h_ctl, CTL_HOST_WORDS * sizeof(int), cudaMemcpyHostToDevice, c->stream));
    }
    // the whole step depends on (token,pos) only through ctl, which advance_kernel updates, so the
    // same graph is replayed back to back with no host round trip; with several local ranks the
    // launches are interleaved so that no rank's queue runs dry while another's is being filled
    for (int i = 0; i < n_steps; ++i) {
        for (l2b_ctx *c : ranks) {
            if (ranks.size() > 1) L2B_CUDA(ctx, cudaSetDevice(c->device));
            if (c->use_graphs) {
                L2B_CUDA(ctx, cudaGraphLaunch(c->graphs[which], c->stream));
                if (c == ctx) launches += c->launches_per_step + (which == G_PREFILL_LOOP ? 0 : 1);
            } else {
                c->last_launches = 0;
                rc = enqueue_call(c, c->stream, which);
                if (rc) { ctx->err = c->err; return rc; }
                if (c == ctx) launches += c->last_launches;
            }
        }
    }
    for (l2b_ctx *c : ranks) {
        L2B_CUDA(ctx, cudaSetDevice(c->device));
        if (c == ctx) {
            L2B_CUDA(ctx, cudaMemcpyAsync(c->h_gen, c->gen_out, (size_t)n_steps * sizeof(int),
                                          cudaMemcpyDeviceToHost, c->stream));
            L2B_CUDA(ctx, cudaMemcpyAsync(c->h_ints + 1, c->gen_ndone, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        }
        L2B_CUDA(ctx, cudaMemcpyAsync(c->h_ctl + CTL_WORDS, c->ctl, CTL_WORDS * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        if (c == ctx) L2B_CUDA(ctx, cudaEventRecord(c->ev1, c->stream));
    }
    rc = finish_call(ctx, ranks);
    if (rc) return rc;
    L2B_CUDA(ctx, cudaSetDevice(ctx->device));
    L2B_CUDA(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
    *done_out = ctx->h_ints[1];
    ctx->last_launches = launches;
    if (pos + *done_out > ctx->n_appended) ctx->n_appended = pos + *done_out;
    return L2B_OK;
}

int32_t l2b_generate_argmax(l2b_ctx *ctx, int32_t token, int32_t pos, int32_t n_steps,
                            const int32_t *forced, int32_t stop_on_bos, int32_t *out_next,
                            int32_t *n_done) {
    int rc = check_step_args(ctx, token, pos);
    if (rc) return rc;
    if (!out_next || !n_done || n_steps < 0) return fail(ctx, L2B_ERR_INVALID_ARG, "bad generate arguments");
    if (n_steps > ctx->cfg.seq_len - pos) n_steps = ctx->cfg.seq_len - pos;   // :992-993
    *n_done = 0;
    if (n_steps == 0) return L2B_OK;
    int done = 0;
    rc = run_device_loop(ctx, G_ARGMAX_LOOP, token, pos, n_steps, forced, stop_on_bos, &done);
    if (rc) return rc;
    for (int i = 0; i < done; ++i) out_next[i] = ctx->h_gen[i];
    *n_done = done;
    return L2B_OK;
}

// Prompt prefill (SURVEY 8f.2; src/main.zig:996-1000 feeds prompt tokens through transformer() one
// at a time and throws their logits away).  All positions run back to back on the device with
// the next token forced, the classifier (60 % of stories15M's bytes) is skipped for every position
// whose logits nobody reads, and no position pays a host round trip.  On bandwidth-bound shapes
// (llama2-7B on one GPU) PF_MAXB = 4 positions additionally share each pass over the weights
// (csrc/l2b_prefill.cuh).  Per (row, position) the arithmetic is the decode step's own.
int32_t l2b_prefill(l2b_ctx *ctx, const int32_t *tokens, int32_t n_tokens, int32_t pos0, float *host_logits) {
    if (!ctx || !tokens || n_tokens <= 0) return fail(ctx, L2B_ERR_INVALID_ARG, "bad prefill arguments");
    int rc = check_step_args(ctx, tokens[0], pos0);
    if (rc) return rc;
    if (pos0 + n_tokens > ctx->cfg.seq_len) return fail(ctx, L2B_ERR_INVALID_ARG, "prompt runs past seq_len");
    for (int i = 0; i < n_tokens; ++i)
        if (tokens[i] < 0 || tokens[i] >= ctx->cfg.vocab_size) return fail(ctx, L2B_ERR_INVALID_ARG, "token out of range");
    const int n_silent = host_logits ? n_tokens - 1 : n_tokens;   // positions whose logits are dropped
    rc = pf_prepare(ctx);
    if (rc) return rc;
    if (n_silent > 0 && ctx->pf_ok) {
        // bandwidth-bound shapes: PF_MAXB positions share each pass over the weights
        rc = prefill_batched(ctx, tokens, n_silent, pos0);
        if (rc) return rc;
    } else if (n_silent > 0) {
        std::vector<int32_t> forced(n_silent);
        for (int i = 0; i < n_silent; ++i) forced[i] = tokens[i + 1 < n_tokens ? i + 1 : i];
        int done = 0;
        rc = run_device_loop(ctx, G_PREFILL_LOOP, tokens[0], pos0, n_silent, forced.data(), 0, &done);
        if (rc) return rc;
        if (done != n_silent) return fail(ctx, L2B_ERR_STATE, "prefill stopped early");
    }
    if (host_logits) return l2b_forward(ctx, tokens[n_tokens - 1], pos0 + n_tokens - 1, host_logits);
    return L2B_OK;
}

// ---- decode streams over one copy of the weights --------------------------------------------------
int32_t l2b_create_stream(l2b_ctx **out, l2b_ctx *base) {
    if (!out || !base) { g_create_error = "NULL argument"; return L2B_ERR_INVALID_ARG; }
    *out = nullptr;
    if (base->world > 1 || base->leader || !base->members.empty() || !base->weights) {
        g_create_error = "decode streams share the weights of a single-GPU context only";
        return fail(base, L2B_ERR_UNSUPPORTED, "decode streams share the weights of a single-GPU context only");
    }
    l2b_ctx *ctx = new l2b_ctx();
    int rc = open_rank(ctx, &base->cfg, 0, 1, base->device, base->num_sms);
    if (rc == L2B_OK) {
        ctx->weights = base->weights;       // no upload: load_bytes stays 0
        ctx->emb = base->emb; ctx->rms_att = base->rms_att; ctx->rms_ffn = base->rms_ffn; ctx->rms_final = base->rms_final;
        ctx->wq = base->wq; ctx->wk = base->wk; ctx->wv = base->wv; ctx->wo = base->wo;
        ctx->w1 = base->w1; ctx->w2 = base->w2; ctx->w3 = base->w3; ctx->wcls = base->wcls;
        rc = init_run_state(ctx, nullptr, nullptr, base);
    }
    if (rc == L2B_OK) rc = warm_up(std::vector<l2b_ctx *>{ctx});
    if (rc) {
        destroy_rank(ctx);
        return rc;
    }
    *out = ctx;
    return L2B_OK;
}

int32_t l2b_forward_batch(l2b_ctx *const *streams, int32_t n, const int32_t *tokens, const int32_t *pos,
                          float *host_logits) {
    int rc = check_batch_args(streams, n, tokens, pos);
    if (rc) return rc;
    l2b_ctx *lead = streams[0];
    if (!host_logits) return fail(lead, L2B_ERR_INVALID_ARG, "host_logits is NULL");
    if ((rc = pf_prepare(lead))) return rc;
    if (lead->pf_ok) return run_batch(streams, n, tokens, pos, 1, nullptr, 0, host_logits, nullptr, nullptr);
    // latency-bound shapes: each stream's own step in turn
    const size_t V = lead->cfg.vocab_size;
    float ms = 0.0f;
    int launches = 0;
    for (int k = 0; k < n; ++k) {
        rc = l2b_forward(streams[k], tokens[k], pos[k], host_logits + (size_t)k * V);
        if (rc) { if (k) lead->err = streams[k]->err; return rc; }
        ms += streams[k]->last_ms; launches += streams[k]->last_launches;
    }
    lead->last_ms = ms; lead->last_launches = launches;
    return L2B_OK;
}

int32_t l2b_generate_argmax_batch(l2b_ctx *const *streams, int32_t n, const int32_t *tokens, const int32_t *pos,
                                  int32_t n_steps, const int32_t *forced, int32_t stop_on_bos, int32_t *out_next,
                                  int32_t *n_done) {
    int rc = check_batch_args(streams, n, tokens, pos);
    if (rc) return rc;
    l2b_ctx *lead = streams[0];
    if (!out_next || !n_done || n_steps < 0) return fail(lead, L2B_ERR_INVALID_ARG, "bad generate arguments");
    if ((rc = pf_prepare(lead))) return rc;
    if (lead->pf_ok) return run_batch(streams, n, tokens, pos, n_steps, forced, stop_on_bos, nullptr, out_next, n_done);
    float ms = 0.0f;
    int launches = 0;
    for (int k = 0; k < n; ++k) {
        rc = l2b_generate_argmax(streams[k], tokens[k], pos[k], n_steps, forced ? forced + (size_t)k * n_steps : nullptr,
                                 stop_on_bos, out_next + (size_t)k * n_steps, &n_done[k]);
        if (rc) { if (k) lead->err = streams[k]->err; return rc; }
        if (n_done[k] > 0) { ms += streams[k]->last_ms; launches += streams[k]->last_launches; }
    }
    lead->last_ms = ms; lead->last_launches = launches;
    return L2B_OK;
}

int32_t l2b_read_state(l2b_ctx *ctx, int32_t which, float *dst, uint64_t n, uint64_t *n_out) {
    if (!ctx || !dst) return L2B_ERR_INVALID_ARG;
    const float *src = nullptr;
    uint64_t cnt = 0;
    const uint64_t L = ctx->cfg.n_layers, S = ctx->cfg.seq_len;
    switch (which) {
    case 0: src = ctx->final_X ? ctx->final_X : ctx->X; cnt = ctx->dim; break;
    case 1: src = ctx->xb; cnt = ctx->q_loc; break;
    case 2: src = ctx->hb; cnt = ctx->hid_loc; break;
    case 3: src = ctx->q; cnt = ctx->q_loc; break;
    case 4: src = ctx->kcache; cnt = L * S * ctx->kv_loc; break;
    case 5: src = ctx->vcache; cnt = L * S * ctx->kv_loc; break;
    case 6: src = ctx->logits; cnt = ctx->cfg.vocab_size; break;
    default: return fail(ctx, L2B_ERR_INVALID_ARG, "unknown state id");
    }
    if (n < cnt) return fail(ctx, L2B_ERR_INVALID_ARG, "dst too small");
    L2B_CUDA(ctx, cudaSetDevice(ctx->device));
    L2B_CUDA(ctx, cudaMemcpy(dst, src, cnt * sizeof(float), cudaMemcpyDeviceToHost));
    if (n_out) *n_out = cnt;
    return L2B_OK;
}

int32_t l2b_last_timing(const l2b_ctx *ctx, float *device_ms, int32_t *kernel_launches) {
    if (!ctx) return L2B_ERR_INVALID_ARG;
    if (device_ms) *device_ms = ctx->last_ms;
    if (kernel_launches) *kernel_launches = ctx->last_launches;
    return L2B_OK;
}

int32_t l2b_load_stats(const l2b_ctx *ctx, double *upload_ms, uint64_t *upload_bytes) {
    if (!ctx) return L2B_ERR_INVALID_ARG;
    if (upload_ms) *upload_ms = ctx->load_ms;
    if (upload_bytes) *upload_bytes = ctx->load_bytes;
    return L2B_OK;
}

int32_t l2b_profile_step(l2b_ctx *ctx, int32_t token, int32_t pos, l2b_kernel_time *out, int32_t cap,
                         int32_t *n_out) {
    int rc = check_step_args(ctx, token, pos);
    if (rc) return rc;
    if (!out || !n_out || cap <= 0) return fail(ctx, L2B_ERR_INVALID_ARG, "bad profile arguments");
    std::vector<l2b_ctx *> ranks = locals(ctx);
    if (pos + 1 > ctx->n_appended) ctx->n_appended = pos + 1;   // attention bytes use this
    const int saved_appended = ctx->n_appended;
    cudaEvent_t last = nullptr;
    for (l2b_ctx *c : ranks) {
        L2B_CUDA(ctx, cudaSetDevice(c->device));
        c->n_appended = pos + 1;
        fill_ctl(c, token, pos, 0, 1.0f, -1.0f);
        L2B_CUDA(ctx, cudaMemcpyAsync(c->ctl, c->h_ctl, CTL_HOST_WORDS * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        c->profiling = (c == ctx);
        c->prof_ev.clear();
        c->prof_rec.clear();
        int r2 = enqueue_step(c, c->stream, MODE_LOGITS);
        c->profiling = false;
        if (r2 && rc == L2B_OK) { rc = r2; ctx->err = c->err; }
        if (c == ctx && rc == L2B_OK) {
            if (cudaEventCreate(&last) != cudaSuccess || cudaEventRecord(last, c->stream) != cudaSuccess)
                rc = fail(ctx, L2B_ERR_CUDA, "event record failed");
        }
        cudaMemcpyAsync(c->h_ctl + CTL_WORDS, c->ctl, CTL_WORDS * sizeof(int), cudaMemcpyDeviceToHost, c->stream);
    }
    ctx->n_appended = saved_appended;
    {
        int r2 = finish_call(ctx, ranks);
        if (rc == L2B_OK) rc = r2;
    }
    cudaSetDevice(ctx->device);
    const int n = (int)ctx->prof_rec.size();
    if (rc == L2B_OK) {
        for (int i = 0; i < n; ++i) {
            cudaEvent_t b = (i + 1 < n) ? ctx->prof_ev[i + 1] : last;
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, ctx->prof_ev[i], b);
            ctx->prof_rec[i].ms = ms;
            if (i < cap) out[i] = ctx->prof_rec[i];
        }
        *n_out = n;
    }
    for (cudaEvent_t e : ctx->prof_ev) cudaEventDestroy(e);
    if (last) cudaEventDestroy(last);
    ctx->prof_ev.clear();
    return rc;
}

// debug: copy the in-kernel timeline of the last step (L2B_TRACE=1) to the host
int32_t l2b_debug_trace(l2b_ctx *ctx, unsigned long long *dst, uint64_t cap_words, uint64_t *n_words) {
    if (!ctx || !dst) return L2B_ERR_INVALID_ARG;
    if (!ctx->trace) return fail(ctx, L2B_ERR_STATE, "tracing not enabled (L2B_TRACE=1)");
    const uint64_t n = (uint64_t)ctx->trace_launches * TRACE_MAX_CTAS * TRACE_SLOTS;
    if (cap_words < n) return fail(ctx, L2B_ERR_INVALID_ARG, "dst too small");
    L2B_CUDA(ctx, cudaSetDevice(ctx->device));
    L2B_CUDA(ctx, cudaMemcpy(dst, ctx->trace, n * 8, cudaMemcpyDeviceToHost));
    if (n_words) *n_words = n;
    return L2B_OK;
}

int32_t l2b_step_bytes(const l2b_ctx *ctx, int32_t pos, uint64_t *weight_bytes, uint64_t *kv_bytes) {
    if (!ctx) return L2B_ERR_INVALID_ARG;
    const uint64_t dim = ctx->dim, L = ctx->cfg.n_layers;
    // SURVEY.md 8d: every weight touched once per token (+ the embedding row), this rank's shard
    uint64_t w = L * ((uint64_t)ctx->q_loc * dim + 2ull * ctx->kv_loc * dim + dim * ctx->q_loc +
                      3ull * ctx->hid_loc * dim + 2 * dim) +
                 dim + (uint64_t)ctx->vocab_loc * dim;
    if (weight_bytes) *weight_bytes = 4 * w;
    if (kv_bytes) *kv_bytes = 4ull * L * 2 * ctx->kv_loc * (uint64_t)(pos + 1);
    return L2B_OK;
}

int32_t l2b_comm_unique_id(uint8_t id[128]) {
    if (!id) return L2B_ERR_INVALID_ARG;
    std::string e;
    if (!nccl_load(&e)) { g_create_error = e; return L2B_ERR_COMM; }
    ncclUniqueId u;
    if (g_nccl.GetUniqueId(&u) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return L2B_ERR_COMM; }
    memcpy(id, &u, 128);
    return L2B_OK;
}

// ---- synthetic generator, host mirror ------------------------------------------------------
void l2b_synth_fill_host(float *dst, uint64_t first, uint64_t count, uint64_t tensor_seed, double mean,
                         double sigma, float lo, float hi) {
    const double scale = sigma * kSynthInvStd;
    for (uint64_t j = 0; j < count; ++j) {
        const int32_t s = synth_irwin_hall(tensor_seed, first + j);
        volatile double prod = (double)s * scale;   // no a*b+c contraction
        float v = (float)(prod + mean);
        v = fminf(fmaxf(v, lo), hi);
        dst[j] = v;
    }
}

int32_t l2b_synth_checkpoint_host(const l2b_config *cfg, uint64_t seed, float *data, uint64_t n_floats) {
    if (!cfg || !data) return L2B_ERR_INVALID_ARG;
    if (n_floats < checkpoint_floats(cfg)) return L2B_ERR_INVALID_ARG;
    const uint64_t dim = cfg->dim, hid = cfg->hidden_dim, L = cfg->n_layers, V = cfg->vocab_size, S = cfg->seq_len;
    const uint64_t hs = dim / cfg->n_heads, kvd = hs * cfg->n_kv_heads;
    const double sd = sqrt(288.0 / (double)dim), sh = sqrt(768.0 / (double)hid);
    const float BIG = 3.0e38f;
    float *p = data;
    auto T = [&](int id, uint64_t count, double mean, double sigma, float lo, float hi) {
        l2b_synth_fill_host(p, 0, count, mix64(seed * 1000003ull + (uint64_t)id), mean, sigma, lo, hi);
        p += count;
    };
    T(1, V * dim, 0.0, 0.04, -BIG, BIG);
    T(2, L * dim, 1.35, 0.35, 0.25f, 2.4f);
    T(3, L * dim * dim, 0.0, 0.04 * sd, -BIG, BIG);
    T(4, L * kvd * dim, 0.0, 0.04 * sd, -BIG, BIG);
    T(5, L * kvd * dim, 0.0, 0.02 * sd, -BIG, BIG);
    T(6, L * dim * dim, 0.0, 0.02 * sd, -BIG, BIG);
    T(7, L * dim, 1.35, 0.35, 0.25f, 2.4f);
    T(8, L * hid * dim, 0.0, 0.026 * sd, -BIG, BIG);
    T(9, L * dim * hid, 0.0, 0.026 * sh, -BIG, BIG);
    T(10, L * hid * dim, 0.0, 0.026 * sd, -BIG, BIG);
    T(11, dim, 7.1, 0.6, 3.0f, 10.0f);
    memset(p, 0, sizeof(float) * 2 * (S * hs / 2));
    p += 2 * (S * hs / 2);
    if (!cfg->shared_weights) T(14, V * dim, 0.0, 0.04, -BIG, BIG);
    return L2B_OK;
}

// ---- single ops with host buffers (unit-test surface) ----------------------------------------
namespace {
struct OpScope {
    int rc = L2B_OK;
    std::vector<void *> bufs;
    explicit OpScope(int device) {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); rc = L2B_ERR_NO_DEVICE; g_create_error = "no CUDA device"; return; }
        if (device < 0 || device >= ndev) { rc = L2B_ERR_INVALID_ARG; g_create_error = "device out of range"; return; }
        if (cudaSetDevice(device) != cudaSuccess) { rc = L2B_ERR_CUDA; g_create_error = "cudaSetDevice failed"; }
    }
    float *up(const float *h, size_t n) {
        if (rc) return nullptr;
        void *d = nullptr;
        if (cudaMalloc(&d, (n ? n : 1) * sizeof(float)) != cudaSuccess) { rc = L2B_ERR_OOM; g_create_error = "cudaMalloc failed"; return nullptr; }
        bufs.push_back(d);
        if (h && cudaMemcpy(d, h, n * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) { rc = L2B_ERR_CUDA; g_create_error = "H2D failed"; }
        return (float *)d;
    }
    void down(float *h, const float *d, size_t n) {
        if (rc) return;
        cudaError_t e = cudaDeviceSynchronize();
        if (e == cudaSuccess) e = cudaMemcpy(h, d, n * sizeof(float), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { rc = L2B_ERR_CUDA; g_create_error = std::string("op failed: ") + cudaGetErrorString(e); }
    }
    ~OpScope() { for (void *p : bufs) cudaFree(p); }
};
}  // namespace

// W . rmsnorm(x, gamma) (gamma NULL => W . x), optionally accumulated into resid_inout, through a
// chosen GEMV kernel flavour: the fused prologue / residual epilogue of the hot path in isolation
int32_t l2b_op_fused_matmul(int32_t device, float *xout, const float *x, const float *gamma, const float *w,
                            float *resid_inout, int32_t d, int32_t n, int32_t kernel) {
    if ((!xout && !resid_inout) || !x || !w || d <= 0 || n <= 0 || kernel < 0 || kernel > 3) return L2B_ERR_INVALID_ARG;
    if (n % 4) { g_create_error = "n must be a multiple of 4"; return L2B_ERR_UNSUPPORTED; }
    OpScope s(device);
    float *dx = s.up(x, n), *dw = s.up(w, (size_t)d * n), *dg = gamma ? s.up(gamma, n) : nullptr;
    float *dout = s.up(resid_inout ? resid_inout : nullptr, d);
    int *ctl = (int *)s.up(nullptr, CTL_WORDS);
    if (s.rc) return s.rc;
    cudaMemset(ctl, 0, CTL_WORDS * sizeof(int));
    l2b_ctx tmp;   // only for launch_gemv's bookkeeping
    tmp.device = device;
    tmp.force_kernel = kernel;
    cudaDeviceProp prop{};
    cudaGetDeviceProperties(&prop, device);
    tmp.num_sms = prop.multiProcessorCount;
    GemvParams p{};
    p.ctl = ctl; p.n = n; p.x_in = dx; p.gamma = dg; p.w0 = dw; p.total_rows = d; p.rows0 = d; p.out0 = dout;
    int rc = launch_gemv(&tmp, resid_inout ? EPI_RESID : EPI_STORE, p, 0);
    if (rc) { g_create_error = tmp.err; return rc; }
    s.down(resid_inout ? resid_inout : xout, dout, d);
    return s.rc;
}

int32_t l2b_op_matmul(int32_t device, float *xout, const float *x, const float *w, int32_t d, int32_t n) {
    if (!xout || !x || !w || d <= 0 || n <= 0) return L2B_ERR_INVALID_ARG;   // asserts :534-536
    if (n % 4 == 0) return l2b_op_fused_matmul(device, xout, x, nullptr, w, nullptr, d, n, 0);
    OpScope s(device);
    float *dx = s.up(x, n), *dw = s.up(w, (size_t)d * n), *dout = s.up(nullptr, d);
    if (s.rc) return s.rc;
    int blocks = (d + NWARP - 1) / NWARP;
    gemv_scalar_kernel<<<blocks, NT>>>(dout, dx, dw, d, n);
    s.down(xout, dout, d);
    return s.rc;
}

int32_t l2b_op_rmsnorm(int32_t device, float *o, const float *x, const float *w, int32_t n) {
    if (!o || !x || !w || n <= 0) return L2B_ERR_INVALID_ARG;
    OpScope s(device);
    float *dx = s.up(x, n), *dw = s.up(w, n), *dout = s.up(nullptr, n);
    if (s.rc) return s.rc;
    rmsnorm_kernel<<<1, NT>>>(dout, dx, dw, n);
    s.down(o, dout, n);
    return s.rc;
}

int32_t l2b_op_softmax(int32_t device, float *x, int32_t n) {
    if (!x || n <= 0) return L2B_ERR_INVALID_ARG;   // assert :688
    OpScope s(device);
    float *dx = s.up(x, n);
    if (s.rc) return s.rc;
    softmax_kernel<<<1, NT>>>(dx, n);
    s.down(x, dx, n);
    return s.rc;
}

int32_t l2b_op_weighted_sum_rows(int32_t device, float *xout, int32_t out_len, const float *rows,
                                 int32_t row_stride, const float *weights, int32_t n_weights) {
    if (!xout || !rows || !weights || out_len <= 0 || n_weights <= 0 || row_stride < out_len)
        return L2B_ERR_INVALID_ARG;   // asserts :658-661
    OpScope s(device);
    const size_t nrows = (size_t)(n_weights - 1) * row_stride + out_len;
    float *dr = s.up(rows, nrows), *dw = s.up(weights, n_weights), *dout = s.up(nullptr, out_len);
    if (s.rc) return s.rc;
    weighted_rows_kernel<<<(out_len + NT - 1) / NT, NT>>>(dout, out_len, dr, row_stride, dw, n_weights);
    s.down(xout, dout, out_len);
    return s.rc;
}

int32_t l2b_op_attention_head(int32_t device, float *out, const float *q, const float *keys,
                              const float *values, int32_t head_size, int32_t kv_stride, int32_t n_pos) {
    if (!out || !q || !keys || !values || head_size <= 0 || n_pos <= 0 || kv_stride < head_size)
        return L2B_ERR_INVALID_ARG;
    if (head_size % 4 || kv_stride % 4 || head_size > NT) { g_create_error = "head_size/kv_stride must be multiples of 4 and head_size <= 256"; return L2B_ERR_UNSUPPORTED; }
    OpScope s(device);
    const size_t nkv = (size_t)n_pos * kv_stride;
    float *dq = s.up(q, head_size), *dk = s.up(keys, nkv), *dv = s.up(values, nkv), *dout = s.up(nullptr, head_size);
    const int nsplit = n_pos > 256 ? 4 : 1;
    float *po = s.up(nullptr, (size_t)nsplit * head_size), *pml = s.up(nullptr, (size_t)nsplit * 2);
    unsigned int *cnt = (unsigned int *)s.up(nullptr, 1);
    int *ctl = (int *)s.up(nullptr, CTL_WORDS);
    if (s.rc) return s.rc;
    int hctl[CTL_WORDS] = {0, n_pos - 1};
    cudaMemcpy(ctl, hctl, sizeof hctl, cudaMemcpyHostToDevice);
    cudaMemset(cnt, 0, sizeof(unsigned int));
    AttnParams a{};
    a.ctl = ctl; a.q = dq; a.kcache = dk; a.vcache = dv; a.xb = dout; a.part_o = po; a.part_ml = pml;
    a.counters = cnt; a.head_size = head_size; a.kv_dim = kv_stride; a.kv_mul = 1; a.nsplit = nsplit;
    a.min_chunk = 64;
    a.vec = nullptr;                 // single position from the control block
    a.seq_len = n_pos;
    int cap = (n_pos + nsplit - 1) / nsplit;
    if (cap < 64) cap = 64;
    const int G = NT / (head_size / 4);
    const size_t smem = ((size_t)G * head_size + cap) * sizeof(float);
    if (smem > (size_t)kMaxDynSmem) { g_create_error = "n_pos too large"; return L2B_ERR_UNSUPPORTED; }
    cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem);
    {
        const char *enva = getenv("L2B_ATTN");
        size_t smem2 = smem;
        attn_fn fn = pick_attention(head_size, !(enva && strcmp(enva, "3pass") == 0), &smem2);
        fn<<<dim3(1, nsplit), NT, smem2>>>(a);
    }
    s.down(out, dout, head_size);
    return s.rc;
}

// sampler preparation alone (src/main.zig:1005-1008, :761-768) on host logits: unit-test surface
int32_t l2b_op_sample_prep(int32_t device, float *logits_inout, int32_t n, float temperature, float top_p,
                           l2b_prob_index *cand, int32_t cand_cap, int32_t *n_cand) {
    if (!logits_inout || n <= 1 || !(temperature > 0.0f) || !n_cand) return L2B_ERR_INVALID_ARG;
    OpScope s(device);
    float *dl = s.up(logits_inout, n);
    int *ctl = (int *)s.up(nullptr, CTL_WORDS);
    ProbIndex *dc = (ProbIndex *)s.up(nullptr, (size_t)2 * (cand_cap > 0 ? cand_cap : 1));
    int *dn = (int *)s.up(nullptr, 1);
    if (s.rc) return s.rc;
    const bool filter = (top_p != 0.0f && top_p != 1.0f);
    const float tp = filter ? top_p : -1.0f;
    int hctl[CTL_WORDS] = {0};
    memcpy(&hctl[CTL_TEMP], &temperature, sizeof(float));
    memcpy(&hctl[CTL_TOPP], &tp, sizeof(float));
    cudaMemcpy(ctl, hctl, sizeof hctl, cudaMemcpyHostToDevice);
    cudaMemset(dn, 0, sizeof(int));
    sample_prep_kernel<<<1, SAMP_THREADS>>>(dl, n, ctl, dc, cand_cap, dn);
    s.down(logits_inout, dl, n);
    if (s.rc) return s.rc;
    int hn = 0;
    cudaMemcpy(&hn, dn, sizeof(int), cudaMemcpyDeviceToHost);
    *n_cand = hn;
    if (filter && cand && hn > 0) {
        const int m = hn < cand_cap ? hn : cand_cap;
        cudaMemcpy(cand, dc, (size_t)m * sizeof(ProbIndex), cudaMemcpyDeviceToHost);
    }
    return s.rc;
}

}  // extern "C"
