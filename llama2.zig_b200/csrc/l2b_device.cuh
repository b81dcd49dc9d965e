// l2b_device.cuh — sm_100a device building blocks for the llama2.zig decode step.
//
// Everything here is fp32 and HBM/L2-bandwidth bound (batch-1 decode is a vector
// contraction: 0.5 flop per weight byte), so there is deliberately no tensor-core code.
// What matters on B200 for this path: 128-bit coalesced streaming loads with many of them
// in flight per SM, the activation vector staged once per CTA into shared memory by a TMA
// bulk copy (cp.async.bulk + mbarrier), persistent CTAs sized from the SM count, and
// warp-shuffle reductions.
#pragma once

#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace l2b {

constexpr int NT = 256;          // threads per CTA for every kernel in this file
constexpr int NWARP = NT / 32;
constexpr int GEMV_R = 2;        // weight rows per thread-group (pairs: RoPE (i,i+1), SiLU (w1,w3))
constexpr int GEMV_U = 4;        // 128-bit loads per row per chunk => R*U = 8 loads in flight/thread

// ---------------------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// Streaming 128-bit load of immutable weights: read-only path, do not allocate in L1.
__device__ __forceinline__ float4 ldg_stream(const float4 *p) {
    float4 r;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
        : "l"(p));
    return r;
}

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    // make the init visible to the async (TMA) proxy
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier.
// dst, src 16-byte aligned; bytes a multiple of 16.  SASS: UBLKCP.
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes,
                                            uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-
// serialization attribute may start while its predecessor is still running; everything before
// pdl_wait() (barrier init, prefetch of immutable weights) overlaps the predecessor's tail.
// pdl_wait() returns once the predecessor grid has completed and its writes are visible.
__device__ __forceinline__ void pdl_launch_dependents() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------
// Tensor-parallel exchange over NVLink peer memory: "LL" units (the low-latency protocol shape
// NCCL uses for small messages).  A value travels as an 8-byte unit {fp32 bits, epoch flag}; two
// units go out as one 16-byte posted store.  8-byte aligned 8-byte stores land atomically, so a
// receiver that sees flag == epoch also sees the value: no fence, no separate signal, one NVLink
// one-way trip.  `epoch` = number of decode steps started on the context (ctl[CTL_EPOCH], >= 1;
// landing buffers start zeroed), identical on every rank because ranks step in lockstep.
// ---------------------------------------------------------------------------------------
constexpr int MAX_TP = 8;
__device__ __forceinline__ void ll_store2(unsigned long long *dst_unit, float a, float b, unsigned int epoch) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(dst_unit), "r"(__float_as_uint(a)),
                 "r"(epoch), "r"(__float_as_uint(b)), "r"(epoch)
                 : "memory");
}
__device__ __forceinline__ uint4 ll_load2(const unsigned long long *src_unit) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(src_unit)
                 : "memory");
    return v;
}
__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned int *p, unsigned int v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_global() {
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
__device__ __forceinline__ unsigned long long global_ns();
// Bounded spin: a dead or diverged peer must not hang the GPU.  Every 256 polls the waiter looks at
// the clock and at ctl[CTL_ERR]; on timeout it raises CTL_ERR (the host turns that into
// L2B_ERR_COMM after the step) and every later wait of the step returns at once.
struct SpinGuard {
    int *ctl;
    unsigned long long t0, limit_ns;
    unsigned int polls;
    __device__ __forceinline__ bool expired();
};

// Optional in-kernel timeline (L2B_TRACE=1): %globaltimer stamps per CTA, 8 slots per CTA.
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
constexpr int TRACE_SLOTS = 8, TRACE_MAX_CTAS = 512;
#define L2B_STAMP(tr, slot) do { if (tr) (tr)[(size_t)blockIdx.x * TRACE_SLOTS + (slot)] = global_ns(); } while (0)

// ---------------------------------------------------------------------------------------
// Block-level reductions (warp shuffles + one smem hop).  Result returned to all threads.
// scratch: >= NWARP + 1 floats of shared memory.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float block_sum(float v, float *scratch) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();  // scratch may still be read from a previous reduction
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    float t = (lane < NWARP) ? scratch[lane] : 0.0f;
    t = warp_sum(t);
    return t;
}
__device__ __forceinline__ float block_max(float v, float *scratch) {
    v = warp_max(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) scratch[w] = v;
    __syncthreads();
    float t = (lane < NWARP) ? scratch[lane] : -INFINITY;
    t = warp_max(t);
    return t;
}

__device__ __forceinline__ float dot4(const float4 a, const float4 b, float acc) {
    acc = fmaf(a.x, b.x, acc);
    acc = fmaf(a.y, b.y, acc);
    acc = fmaf(a.z, b.z, acc);
    acc = fmaf(a.w, b.w, acc);
    return acc;
}

// Orderable key for a device-side argmax with the reference's tie rule (src/main.zig:715-726:
// strict '>' so the FIRST maximum wins): larger value wins, then smaller index.
__device__ __forceinline__ unsigned long long argmax_key(float v, int idx) {
    uint32_t u = __float_as_uint(v);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return (static_cast<unsigned long long>(u) << 32) | (0xFFFFFFFFu - static_cast<uint32_t>(idx));
}

// ---------------------------------------------------------------------------------------
// Step control block (device memory, 16 ints):
//   [0] token  [1] pos  [2] done flag (generation loop saw BOS)  [3] step index in generate
//   [4] stop-on-BOS enabled  [5] sampler temperature, [6] sampler top-p (fp32 bits; top-p < 0 = no
//   candidate filter), consumed by sample_prep_kernel
//   [8] epoch: number of decode steps started on this context (never reset; it is the flag value of
//       the tensor-parallel LL units and the multiplier of the slice counters)
//   [9] error word: a tensor-parallel wait timed out (peer dead or out of lockstep)
// The host writes words [0..7] through a pinned-memory copy at the head of a step graph; words
// [8] and [9] are only ever written by the device.
// ---------------------------------------------------------------------------------------
enum { CTL_TOKEN = 0, CTL_POS = 1, CTL_DONE = 2, CTL_STEP = 3, CTL_STOP_ON_BOS = 4, CTL_TEMP = 5, CTL_TOPP = 6,
       CTL_EPOCH = 8, CTL_ERR = 9, CTL_WORDS = 16, CTL_HOST_WORDS = 8 };

__device__ __forceinline__ bool SpinGuard::expired() {
    if ((++polls & 255u) != 0u) return false;
    if (*reinterpret_cast<volatile int *>(ctl + CTL_ERR)) return true;
    if (global_ns() - t0 > limit_ns) {
        *reinterpret_cast<volatile int *>(ctl + CTL_ERR) = 1;
        return true;
    }
    return false;
}
__device__ __forceinline__ SpinGuard spin_guard(const int *ctl, unsigned long long limit_ns) {
    SpinGuard g;
    g.ctl = const_cast<int *>(ctl);
    g.t0 = global_ns();
    g.limit_ns = limit_ns;
    g.polls = *reinterpret_cast<volatile int *>(g.ctl + CTL_ERR) ? 255u : 0u;   // already failed: give up on the first poll
    return g;
}

// ---------------------------------------------------------------------------------------
// GEMV: out = W(rows, n) . xs(n), W row-major fp32 (src/main.zig:485-498, :530-605).
//
// Work decomposition: a group of TPR threads owns GEMV_R consecutive (virtual) rows and walks
// their columns in 128-bit steps of stride TPR, so a group reads TPR*16 contiguous bytes per
// row per step (fully coalesced, every 128-byte line used whole).  A tile is (NT/TPR)*GEMV_R
// rows; CTAs are persistent and stride over tiles.  Loads of the next chunk are issued before
// the reduction/epilogue of the current one so HBM requests stay in flight across tiles.
//
// Prologue (once per CTA): the input vector (and, when fused, the pending residual delta and
// the RMSNorm gain) are staged into shared memory by TMA bulk copies; optional fused
// rmsnorm (src/main.zig:432-468) with the reference's rounding points (x*s)*w.
// ---------------------------------------------------------------------------------------
enum GemvEpi {
    EPI_STORE = 0,   // out[v] = acc                                   (wcls; :429)
    EPI_ARGMAX = 1,  // EPI_STORE + device argmax                       (:715-726 fused, 8f.1)
    EPI_QKV = 2,     // RoPE on (even,odd) pairs + KV-cache append     (:308-358)
    EPI_SILU = 3,    // hb[i] = silu(w1.x) * (w3.x)                     (:405-416)
    EPI_XCHG = 4,    // tensor parallel: partial rows sent as LL units to every rank's landing area (8e)
    EPI_RESID = 5,   // x[v] += acc: the residual add of :395 / :422 fused into wo / w2
    EPI_COUNT = 6
};

struct GemvParams {
    // ---- input vector / prologue
    const float *x_in;      // n floats; when emb != nullptr: row `token` of emb is used instead
    const float *emb;       // token embedding table (layer 0: x = emb[token], :295-296) or nullptr
    const float *gamma;     // rmsnorm gain (n floats) => fused rmsnorm, or nullptr => plain staging
    float *x_out;           // CTA 0 writes the staged (un-normalised) x here: layer 0 (x = embedding row) and
                            // kernels that fold `parts` in (x_out must then differ from x_in)
    const float *parts;     // small-model fusion: nparts partial vectors [nparts][n] whose fixed-order sum is the
    int nparts;             // pending residual (the wo / w2 result split by head / by hidden slice), or nullptr
    const int *ctl;         // control block (token, pos, done, epoch, error)
    int n;                  // columns (multiple of 4)
    // ---- matrices (virtual row space depends on the epilogue)
    const float *w0, *w1, *w2;
    int rows0, rows1, rows2;  // EPI_QKV: q/k/v rows.  EPI_SILU: rows0 = hidden (virtual rows = 2*hidden)
    int total_rows;           // virtual rows
    // ---- outputs
    float *out0;            // STORE: out; QKV: q; SILU: hb; RESID: the residual stream x (read-modify-write)
    float *kcache, *vcache; // QKV: this layer's (seq_len, kv_dim) caches
    const float *rope_cos, *rope_sin;  // (seq_len, head_size/2)
    int head_size, kv_dim;
    unsigned long long *amax;  // ARGMAX: packed running maximum (must be 0 before the launch)
    int row_base;              // ARGMAX / XCHG: global index of out row 0 (vocab shard offset)
    int nstage;                // gemv_tma_kernel: ring depth (2..TMA_MAX_STAGES)
    int nprefill;              // gemv_tma_kernel: stages put in flight BEFORE the dependency wait (1..nstage)
    // ---- tensor-parallel exchange (fused GEMV + all-reduce over peer memory); unused when ll_ndst == 0
    // EPI_XCHG: row v of my result goes, as an LL unit, to ll_out[d][row_base + v] for every
    // destination d < ll_ndst (the landing area reserved for MY rank on that peer).
    unsigned long long *ll_out[MAX_TP];
    int ll_ndst;
    // All-reduce tail (wo / w2; xres != nullptr): once a CTA has sent its own rows, CTA s < ceil(rows/128)
    // folds slice s of ALL ranks' partial rows (ll_in[r * total_rows + i], they arrive straight from
    // the other CTAs' / other GPUs' epilogues) into the residual stream: xres[i] += sum_r partial_r[i].
    const unsigned long long *ll_in;
    float *xres;
    int xworld;
    int bump_epoch;            // set on the first kernel of a step: CTA 0 increments ctl[CTL_EPOCH]
    unsigned long long spin_ns;  // bound on every peer wait (SpinGuard)
    unsigned long long *trace;   // nullptr or this launch's [grid][TRACE_SLOTS] timeline
};

template <int EPI>
__device__ __forceinline__ const float *gemv_row_ptr(const GemvParams &p, int v) {
    if (EPI == EPI_QKV) {
        if (v < p.rows0) return p.w0 + (size_t)v * p.n;
        v -= p.rows0;
        if (v < p.rows1) return p.w1 + (size_t)v * p.n;
        v -= p.rows1;
        return p.w2 + (size_t)v * p.n;
    } else if (EPI == EPI_SILU) {
        return ((v & 1) ? p.w1 : p.w0) + (size_t)(v >> 1) * p.n;
    } else {
        return p.w0 + (size_t)v * p.n;
    }
}

// ---- tensor-parallel all-reduce, second half, run by ONE warp of a wo / w2 CTA after that CTA has
// sent its own partial rows.  The residual stream x is updated IN PLACE:
//   x[i] += sum_r partial_r[i]   (fixed rank order: every rank forms bit-identical x)
// Work is cut into slices of 32 float4; slice s belongs to CTA (s mod grid), which polls the LL units
// of that slice — they arrive straight from the epilogues of the CTAs (local and, over NVLink,
// remote) that own those rows — and writes the new x slice.  Kernel completion then means "x is
// reduced", so the consumer kernel's prologue is the single-GPU one and stages 16 KB of finished x
// instead of g x 16 KB of partials.  Doing this at the TAIL of the producer rather than in the
// consumer's prologue matters: measured (r02, 2 GPUs), loads issued from a CTA whose TMA ring is
// pre-filling wait ~4 us behind the 192 KB that SM already requested.
constexpr int TP_SLICE4 = 32;
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tp_reduce_tail(const GemvParams &p, unsigned int epoch, int lane) {
    const int n4 = p.total_rows >> 2;
    const int nslices = (n4 + TP_SLICE4 - 1) / TP_SLICE4;
    SpinGuard sg = spin_guard(p.ctl, p.spin_ns);
    float4 *x4 = reinterpret_cast<float4 *>(p.xres);
    for (int s = blockIdx.x; s < nslices; s += gridDim.x) {
        const int i = s * TP_SLICE4 + lane;
        if (i < n4) {
            float4 v = __ldcg(x4 + i);
            // the units of up to four ranks are requested together (measured r02, 8 GPUs: polling rank
            // after rank serialised eight L2 round trips and made this tail 6 us), then re-polled
            // until every flag carries this step's epoch; the sum itself stays in rank order
            for (int rb = 0; rb < p.xworld; rb += 4) {
                uint4 a[4], b[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    a[k] = b[k] = make_uint4(0u, epoch, 0u, epoch);        // ranks beyond the world count as "arrived"
                    if (rb + k < p.xworld) {
                        const unsigned long long *u = p.ll_in + (size_t)(rb + k) * p.total_rows + (size_t)i * 4;
                        a[k] = ll_load2(u);
                        b[k] = ll_load2(u + 2);
                    }
                }
                bool all = false;
                while (!all) {
                    all = true;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (a[k].y != epoch || a[k].w != epoch || b[k].y != epoch || b[k].w != epoch) {
                            const unsigned long long *u = p.ll_in + (size_t)(rb + k) * p.total_rows + (size_t)i * 4;
                            a[k] = ll_load2(u);
                            b[k] = ll_load2(u + 2);
                            all = false;
                        }
                    }
                    if (!all && sg.expired()) break;
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (rb + k < p.xworld) {
                        v.x += __uint_as_float(a[k].x); v.y += __uint_as_float(a[k].z);   // accum(), :708-713
                        v.z += __uint_as_float(b[k].x); v.w += __uint_as_float(b[k].z);
                    }
                }
            }
            __stcg(x4 + i, v);
        }
    }
}

// ---- shared prologue: stage the activation vector (+ rmsnorm) into shared memory.
// Must be called by all NT threads after pdl_wait(); thread 0 has already initialised `bar`.
__device__ __forceinline__ void gemv_stage_input(const GemvParams &p, float *xs, float *aux,
                                                 uint64_t *bar, float *scratch) {
    const int tid = threadIdx.x;
    const int n4 = p.n >> 2;
    const float *xsrc = p.emb ? p.emb + (size_t)p.ctl[CTL_TOKEN] * p.n : p.x_in;
    float *gs = aux;
    float *ps = p.gamma ? aux + p.n : aux;               // sum of the partial vectors (when p.parts)
    if (tid == 0) {
        const uint32_t bytes = (uint32_t)p.n * 4u;
        mbar_expect_tx(bar, bytes * (1u + (p.gamma ? 1u : 0u)));
        tma_load_1d(xs, xsrc, bytes, bar);
        if (p.gamma) tma_load_1d(gs, p.gamma, bytes, bar);
    }
    if (p.parts) {
        // the wo / w2 product arrives split into nparts partial vectors (by head / by hidden slice):
        // complete it in fixed order while the bulk copies are in flight
        const float4 *pp = reinterpret_cast<const float4 *>(p.parts);
        for (int i = tid; i < n4; i += NT) {
            float4 a = __ldcg(pp + i);
            for (int j = 1; j < p.nparts; ++j) {
                const float4 d = __ldcg(pp + (size_t)j * n4 + i);
                a.x += d.x; a.y += d.y; a.z += d.z; a.w += d.w;
            }
            reinterpret_cast<float4 *>(ps)[i] = a;
        }
    }
    __syncthreads();  // barrier init visible to all waiters
    mbar_wait(bar, 0);
    if (p.gamma || p.x_out || p.parts) {
        float4 *xs4 = reinterpret_cast<float4 *>(xs);
        float ssq = 0.0f;
        for (int i = tid; i < n4; i += NT) {
            float4 v = xs4[i];
            if (p.parts) {
                const float4 d = reinterpret_cast<const float4 *>(ps)[i];
                v.x += d.x; v.y += d.y; v.z += d.z; v.w += d.w;   // accum(), :708-713
                xs4[i] = v;
            }
            if (p.x_out && blockIdx.x == 0) reinterpret_cast<float4 *>(p.x_out)[i] = v;
            ssq = fmaf(v.x, v.x, ssq); ssq = fmaf(v.y, v.y, ssq);
            ssq = fmaf(v.z, v.z, ssq); ssq = fmaf(v.w, v.w, ssq);
        }
        if (p.gamma) {
            float ss = block_sum(ssq, scratch);
            ss /= (float)p.n;            // :452
            ss += 1e-5f;                 // :453
            const float s = 1.0f / sqrtf(ss);  // :454
            const float4 *gs4 = reinterpret_cast<const float4 *>(gs);
            for (int i = tid; i < n4; i += NT) {
                float4 v = xs4[i];
                const float4 g = gs4[i];
                v.x = __fmul_rn(__fmul_rn(v.x, s), g.x);   // (x*s)*w, :462
                v.y = __fmul_rn(__fmul_rn(v.y, s), g.y);
                v.z = __fmul_rn(__fmul_rn(v.z, s), g.z);
                v.w = __fmul_rn(__fmul_rn(v.w, s), g.w);
                xs4[i] = v;
            }
        }
        __syncthreads();
    }
}

// ---- shared epilogue for one adjacent pair of virtual rows (v0 even).  `xr` is the pair of
// residual-stream values the caller prefetched for EPI_RESID (ignored otherwise).
template <int EPI>
__device__ __forceinline__ void gemv_epilogue_pair(const GemvParams &p, int v0, float a0, float a1,
                                                   int pos, unsigned long long &best, unsigned int epoch,
                                                   float2 xr) {
    if (v0 >= p.total_rows) return;
    if (EPI == EPI_XCHG) {
        // my partial of rows (v0, v0+1) goes to every destination over NVLink as one 16-byte posted
        // store of two LL units (total_rows is even for every exchanged shape: dim % 4 == 0)
        for (int d = 0; d < p.ll_ndst; ++d) ll_store2(p.ll_out[d] + p.row_base + v0, a0, a1, epoch);
    } else if (EPI == EPI_RESID) {
        // accum(), :708-713, applied by the producer: each row of x has exactly one owner
        if (v0 + 1 < p.total_rows) *reinterpret_cast<float2 *>(p.out0 + v0) = make_float2(xr.x + a0, xr.y + a1);
        else p.out0[v0] = xr.x + a0;
    } else if (EPI == EPI_STORE || EPI == EPI_ARGMAX) {
        p.out0[v0] = a0;
        if (v0 + 1 < p.total_rows) p.out0[v0 + 1] = a1;
        if (EPI == EPI_ARGMAX) {
            const unsigned long long k0 = argmax_key(a0, p.row_base + v0);
            best = k0 > best ? k0 : best;
            if (v0 + 1 < p.total_rows) {
                const unsigned long long k1 = argmax_key(a1, p.row_base + v0 + 1);
                best = k1 > best ? k1 : best;
            }
        }
    } else if (EPI == EPI_QKV) {
        // rows (v0, v0+1) are an adjacent pair of q, k or v (segment sizes are even)
        if (v0 < p.rows0 + p.rows1) {
            const bool is_q = v0 < p.rows0;
            const int i = is_q ? v0 : v0 - p.rows0;       // index within q / k
            const int pr = (i % p.head_size) >> 1;          // :338 (i % head_size)
            const float fcr = p.rope_cos[(size_t)pos * (p.head_size >> 1) + pr];
            const float fci = p.rope_sin[(size_t)pos * (p.head_size >> 1) + pr];
            // :348-349, evaluated without FMA contraction like the reference
            const float r0 = __fsub_rn(__fmul_rn(a0, fcr), __fmul_rn(a1, fci));
            const float r1 = __fadd_rn(__fmul_rn(a0, fci), __fmul_rn(a1, fcr));
            float *dst = is_q ? p.out0 + i : p.kcache + (size_t)pos * p.kv_dim + i;   // :355,:357
            *reinterpret_cast<float2 *>(dst) = make_float2(r0, r1);
        } else {
            const int i = v0 - p.rows0 - p.rows1;
            *reinterpret_cast<float2 *>(p.vcache + (size_t)pos * p.kv_dim + i) = make_float2(a0, a1);  // :356,:358
        }
    } else {  // EPI_SILU
        const float sg = __fmul_rn(a0, __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-a0))));   // :412
        p.out0[v0 >> 1] = __fmul_rn(sg, a1);                                          // :416
    }
}

// residual-stream values of rows (v0, v0+1) for EPI_RESID, fetched ahead of the reduction
template <int EPI>
__device__ __forceinline__ float2 gemv_resid_fetch(const GemvParams &p, int v0) {
    float2 r = make_float2(0.f, 0.f);
    if (EPI == EPI_RESID && v0 < p.total_rows) {
        if (v0 + 1 < p.total_rows) r = __ldcg(reinterpret_cast<const float2 *>(p.out0 + v0));
        else r.x = __ldcg(p.out0 + v0);
    }
    return r;
}

template <int EPI>
__device__ __forceinline__ void gemv_finish_argmax(const GemvParams &p, unsigned long long best,
                                                   unsigned long long *blk_key) {
    if (EPI != EPI_ARGMAX) return;
    // CTA-level max, then one 64-bit atomicMax per CTA
    if (threadIdx.x == 0) *blk_key = 0ull;
    __syncthreads();
    if (best) atomicMax(blk_key, best);
    __syncthreads();
    if (threadIdx.x == 0 && *blk_key) atomicMax(p.amax, *blk_key);
}

// ---- v1: small / latency-bound shapes.  TPR threads per pair of rows, tiles strided over CTAs.
template <int TPR, int EPI>
__global__ void __launch_bounds__(NT) gemv_kernel(const GemvParams p) {
    constexpr int GROUPS = NT / TPR;           // row groups per CTA
    constexpr int TILE_ROWS = GROUPS * GEMV_R;
    constexpr int WPG = (TPR + 31) / 32;       // warps per group (TPR > 32)

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *xs = reinterpret_cast<float *>(smem_raw);   // n floats
    float *aux = xs + p.n;                              // delta (n) then gamma (n) when fused
    __shared__ uint64_t bar;
    __shared__ float scratch[NWARP + 1];
    __shared__ float red[NWARP][GEMV_R];
    __shared__ unsigned long long blk_key;

    const int tid = threadIdx.x;
    const int grp = tid / TPR, sub = tid % TPR;
    const int n4 = p.n >> 2;
    const int ntiles = (p.total_rows + TILE_ROWS - 1) / TILE_ROWS;
    const int nchunks = (n4 + TPR * GEMV_U - 1) / (TPR * GEMV_U);

    // ---- first chunk of weights goes in flight before anything that depends on earlier kernels
    float4 wv[GEMV_R][GEMV_U];
    int tile = blockIdx.x, chunk = 0;
    auto issue = [&](int t, int ch) {
        const int v0 = t * TILE_ROWS + grp * GEMV_R;
#pragma unroll
        for (int r = 0; r < GEMV_R; ++r) {
            const int v = v0 + r;
            const bool rok = v < p.total_rows;
            const float4 *wr =
                reinterpret_cast<const float4 *>(gemv_row_ptr<EPI>(p, rok ? v : 0));
#pragma unroll
            for (int u = 0; u < GEMV_U; ++u) {
                const int c = (ch * GEMV_U + u) * TPR + sub;
                wv[r][u] = (rok && c < n4) ? ldg_stream(wr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
    };
    if (tid == 0) L2B_STAMP(p.trace, 0);
    if (tile < ntiles) issue(tile, 0);
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
    }
    bool triggered = false;
    if (tile + (int)gridDim.x >= ntiles && nchunks == 1) {   // this CTA is already on its last chunk
        pdl_launch_dependents();
        triggered = true;
    }

    // ---- everything below reads what earlier kernels of this step wrote
    pdl_wait();
    if (p.ctl[CTL_DONE]) return;  // generation loop already ended (BOS)
    if (p.bump_epoch && blockIdx.x == 0 && tid == 0) const_cast<int *>(p.ctl)[CTL_EPOCH] += 1;
    if (tid == 0) L2B_STAMP(p.trace, 2);
    gemv_stage_input(p, xs, aux, &bar, scratch);
    if (tid == 0) L2B_STAMP(p.trace, 3);

    const float4 *xs4 = reinterpret_cast<const float4 *>(xs);
    const int pos = p.ctl[CTL_POS];
    const unsigned int epoch = (EPI == EPI_XCHG) ? (unsigned int)p.ctl[CTL_EPOCH] : 0u;
    unsigned long long best = 0ull;
    float2 xr = make_float2(0.f, 0.f);
    float acc[GEMV_R];
#pragma unroll
    for (int r = 0; r < GEMV_R; ++r) acc[r] = 0.0f;

    while (tile < ntiles) {
        if (EPI == EPI_RESID && chunk == 0 && sub == 0)   // residual values of this tile's rows, in flight during the dot products
            xr = gemv_resid_fetch<EPI>(p, tile * TILE_ROWS + grp * GEMV_R);
        // ---- consume the chunk in registers
#pragma unroll
        for (int u = 0; u < GEMV_U; ++u) {
            const int c = (chunk * GEMV_U + u) * TPR + sub;
            if (c < n4) {
                const float4 xv = xs4[c];
#pragma unroll
                for (int r = 0; r < GEMV_R; ++r) acc[r] = dot4(wv[r][u], xv, acc[r]);
            }
        }
        // ---- put the next chunk in flight
        int ntile = tile, nchunk = chunk + 1;
        if (nchunk == nchunks) { ntile = tile + gridDim.x; nchunk = 0; }
        if (ntile < ntiles) {
            issue(ntile, nchunk);
        }
        if (!triggered && (ntile >= ntiles || (ntile + (int)gridDim.x >= ntiles && nchunk == nchunks - 1))) {
            pdl_launch_dependents();   // our last chunk is in flight: let the successor start prefetching
            triggered = true;
        }

        if (chunk == nchunks - 1) {
            // ---- reduce the GEMV_R partial dot products across the TPR threads of the group
            if (TPR <= 32) {
#pragma unroll
                for (int r = 0; r < GEMV_R; ++r) {
#pragma unroll
                    for (int o = TPR / 2; o > 0; o >>= 1)
                        acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
                }
            } else {
#pragma unroll
                for (int r = 0; r < GEMV_R; ++r) acc[r] = warp_sum(acc[r]);
                __syncthreads();  // red[] free (previous tile's reads done)
                if ((tid & 31) == 0) {
#pragma unroll
                    for (int r = 0; r < GEMV_R; ++r) red[tid >> 5][r] = acc[r];
                }
                __syncthreads();
                if (sub == 0) {
#pragma unroll
                    for (int r = 0; r < GEMV_R; ++r) {
                        float s = 0.0f;
#pragma unroll
                        for (int w = 0; w < WPG; ++w) s += red[grp * WPG + w][r];
                        acc[r] = s;
                    }
                }
            }
            if (sub == 0)
                gemv_epilogue_pair<EPI>(p, tile * TILE_ROWS + grp * GEMV_R, acc[0], acc[1], pos, best, epoch, xr);
#pragma unroll
            for (int r = 0; r < GEMV_R; ++r) acc[r] = 0.0f;
        }
        tile = ntile;
        chunk = nchunk;
    }
    if (!triggered) pdl_launch_dependents();
    gemv_finish_argmax<EPI>(p, best, &blk_key);
    if (tid == 0) L2B_STAMP(p.trace, 5);
    if (EPI == EPI_XCHG && p.xres && tid < 32) tp_reduce_tail(p, epoch, tid);
    if (tid == 0) L2B_STAMP(p.trace, 7);
}

// ---- v2: bandwidth-bound shapes (n >= 1024, many MB).  The whole CTA (256 threads) walks the
// columns of GEMV8_R = 8 rows at once: per column step one LDS.128 of x is shared by eight
// LDG.128 of weights (32 FMAs), two steps are kept in flight per thread (16 x 128-bit loads),
// and the cross-thread reduction happens once per 8 rows with a transposing butterfly
// (9 shuffles for 8 rows instead of 40) and one barrier.  Each CTA owns a CONTIGUOUS, balanced
// range of row pairs (+-1 pair), so all CTAs stream the same number of bytes and finish together.
constexpr int GEMV8_R = 8;

template <int EPI>
__global__ void __launch_bounds__(NT, 2) gemv8_kernel(const GemvParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *xs = reinterpret_cast<float *>(smem_raw);
    float *aux = xs + p.n;
    __shared__ uint64_t bar;
    __shared__ float scratch[NWARP + 1];
    __shared__ float red[2][NWARP][GEMV8_R];
    __shared__ unsigned long long blk_key;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n4 = p.n >> 2;
    const int nsteps = (n4 + NT - 1) / NT;             // column steps per tile
    // balanced contiguous ranges of row pairs
    const int npairs = (p.total_rows + 1) >> 1;
    const int base = npairs / (int)gridDim.x, rem = npairs % (int)gridDim.x;
    const int b = blockIdx.x;
    const int pair0 = b * base + min(b, rem);
    const int pair1 = pair0 + base + (b < rem ? 1 : 0);
    const int r0 = pair0 * 2, r1 = min(pair1 * 2, p.total_rows);
    const int ntiles = (r1 - r0 + GEMV8_R - 1) / GEMV8_R;
    const int total = ntiles * nsteps;                 // flattened (tile, step) space

    float4 wa[GEMV8_R], wb[GEMV8_R];
    auto issue = [&](float4 (&w)[GEMV8_R], int it) {
        const int t = it / nsteps, st = it - t * nsteps;
        const int c = st * NT + tid;
        const int v0 = r0 + t * GEMV8_R;
#pragma unroll
        for (int r = 0; r < GEMV8_R; ++r) {
            const int v = v0 + r;
            const bool ok = (v < r1) && (c < n4);
            const float4 *wr = reinterpret_cast<const float4 *>(gemv_row_ptr<EPI>(p, ok ? v : 0));
            w[r] = ok ? ldg_stream(wr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    if (0 < total) issue(wa, 0);
    if (1 < total) issue(wb, 1);
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
    }
    bool triggered = false;
    if (total <= 2) { pdl_launch_dependents(); triggered = true; }

    pdl_wait();
    if (p.ctl[CTL_DONE]) return;
    if (p.bump_epoch && blockIdx.x == 0 && tid == 0) const_cast<int *>(p.ctl)[CTL_EPOCH] += 1;
    gemv_stage_input(p, xs, aux, &bar, scratch);

    const float4 *xs4 = reinterpret_cast<const float4 *>(xs);
    const int pos = p.ctl[CTL_POS];
    const unsigned int epoch = (EPI == EPI_XCHG) ? (unsigned int)p.ctl[CTL_EPOCH] : 0u;
    unsigned long long best = 0ull;
    float2 xr = make_float2(0.f, 0.f);
    float acc[GEMV8_R];
#pragma unroll
    for (int r = 0; r < GEMV8_R; ++r) acc[r] = 0.0f;

    auto consume = [&](const float4 (&w)[GEMV8_R], int it) {
        const int t = it / nsteps, st = it - t * nsteps;
        const int c = st * NT + tid;
        if (EPI == EPI_RESID && st == 0 && tid < GEMV8_R / 2)
            xr = gemv_resid_fetch<EPI>(p, (r0 + t * GEMV8_R + 2 * tid < r1) ? r0 + t * GEMV8_R + 2 * tid : p.total_rows);
        if (c < n4) {
            const float4 xv = xs4[c];
#pragma unroll
            for (int r = 0; r < GEMV8_R; ++r) acc[r] = dot4(w[r], xv, acc[r]);
        }
        if (st != nsteps - 1) return;
        // ---- end of a tile: transposing butterfly, lane L (L % 4 == 0) ends with row L / 4
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float send = (lane & 16) ? acc[i] : acc[i + 4];
            const float keep = (lane & 16) ? acc[i + 4] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float send = (lane & 8) ? acc[i] : acc[i + 2];
            const float keep = (lane & 8) ? acc[i + 2] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {
            const float send = (lane & 4) ? acc[0] : acc[1];
            const float keep = (lane & 4) ? acc[1] : acc[0];
            acc[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 2);
        acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
        const int par = t & 1;                         // double-buffered: one barrier per tile
        if ((lane & 3) == 0) red[par][warp][lane >> 2] = acc[0];
        __syncthreads();
        if (tid < GEMV8_R / 2) {
            float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
            for (int w8 = 0; w8 < NWARP; ++w8) {       // fixed order
                s0 += red[par][w8][2 * tid];
                s1 += red[par][w8][2 * tid + 1];
            }
            const int v0 = r0 + t * GEMV8_R + 2 * tid;
            if (v0 < r1) gemv_epilogue_pair<EPI>(p, v0, s0, s1, pos, best, epoch, xr);
        }
#pragma unroll
        for (int r = 0; r < GEMV8_R; ++r) acc[r] = 0.0f;
    };

    for (int it = 0; it < total; it += 2) {
        consume(wa, it);
        if (it + 2 < total) issue(wa, it + 2);
        if (it + 1 < total) {
            consume(wb, it + 1);
            if (it + 3 < total) issue(wb, it + 3);
        }
        if (!triggered && it + 4 >= total) {           // the last loads are in flight
            pdl_launch_dependents();
            triggered = true;
        }
    }
    if (!triggered) pdl_launch_dependents();
    gemv_finish_argmax<EPI>(p, best, &blk_key);
    if (EPI == EPI_XCHG && p.xres && tid < 32) tp_reduce_tail(p, epoch, tid);
}

// ---- v3: TMA-fed streaming GEMV for bandwidth-bound shapes.
//
// Measured on this B200 (profiles/microbench/read_bw.cu): a pure read stream needs ~128 KB in
// flight per SM; register-fed LDG loops only get there with >= 1024 resident threads per SM,
// while a shared-memory ring filled by cp.async.bulk reaches 7.2 TB/s with one small CTA.  So:
// one persistent CTA per SM; a producer thread streams 32 KB stages (8 rows x 256 float4, one
// 4 KB bulk copy per row) of this CTA's contiguous row range into an NSTAGE ring, starting
// BEFORE griddepcontrol.wait (weights are immutable), so the ring is already full when the
// previous kernel finishes; 8 consumer warps read each stage with conflict-free LDS.128, share
// one LDS.128 of x across the 8 rows, and reduce once per 8 rows (transposing butterfly).
__device__ __forceinline__ void prefetch_l2_bulk(const void *p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

constexpr int TMA_MAX_STAGES = 6;                         // ring depth is a launch parameter (GemvParams::nstage)
constexpr int TMA_STAGE_FLOATS = GEMV8_R * NT * 4;        // 8 rows x 256 float4 = 32 KB
constexpr int TMA_THREADS = NT + 64;                       // 8 consumer warps + producer warp + epilogue warp

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Warp roles: warps 0-7 consume stages (LDS.128 + FMA, butterfly reduce per 8 rows), warp 8 lane 0
// produces (TMA), warp 9 runs the epilogues (RoPE / KV append / SiLU / argmax) off the consumers'
// critical path: consumers hand it the 8x8 per-warp partial sums through a double-buffered
// shared array guarded by two mbarrier pairs, so no block-wide barrier exists in the main loop.
template <int EPI>
__global__ void __launch_bounds__(TMA_THREADS, 2) gemv_tma_kernel(const GemvParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NSTAGE = p.nstage;
    float *ring = reinterpret_cast<float *>(smem_raw);                 // NSTAGE x 32 KB
    float *xs = ring + (size_t)NSTAGE * TMA_STAGE_FLOATS;              // n floats
    __shared__ uint64_t full[TMA_MAX_STAGES], empty[TMA_MAX_STAGES], xbar, tile_full[2], tile_free[2];
    __shared__ float scratch[NWARP + 2];
    __shared__ float red[2][NWARP][GEMV8_R];
    __shared__ float rope_s[2][128];                                   // cos/sin row of `pos` (head_size/2 <= 128)

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n4 = p.n >> 2;
    const int nsteps = (n4 + NT - 1) / NT;
    const int npairs = (p.total_rows + 1) >> 1;
    const int base = npairs / (int)gridDim.x, rem = npairs % (int)gridDim.x;
    const int b = blockIdx.x;
    const int pair0 = b * base + min(b, rem);
    const int pair1 = pair0 + base + (b < rem ? 1 : 0);
    const int r0 = pair0 * 2, r1 = min(pair1 * 2, p.total_rows);
    const int ntiles = (r1 - r0 + GEMV8_R - 1) / GEMV8_R;
    const int total = ntiles * nsteps;

    if (tid == 0) {
        L2B_STAMP(p.trace, 0);
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], NWARP); }
        mbar_init(&xbar, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&tile_full[s], NWARP); mbar_init(&tile_free[s], 1); }
        mbar_fence_init();
    }
    __syncthreads();

    // ---- producer state (warp 8): lane r issues row r's bulk copy, lane 0 owns the barriers.
    // The ring is filled before waiting on the previous kernel (weights are immutable).
    int p_it = 0, p_stage = 0, p_tile = 0, p_step = 0;
    uint32_t p_phase = 0;
    const float *p_row = nullptr;                                      // this lane's row in the current tile
    auto produce_one = [&]() {                                         // executed by all 32 lanes of warp 8
        const int c0 = p_step * NT;                                    // first float4 column
        const int cols4 = min(NT, n4 - c0);
        const int v0 = r0 + p_tile * GEMV8_R;
        const int rows = min(GEMV8_R, r1 - v0);
        if (p_step == 0 && lane < rows) p_row = gemv_row_ptr<EPI>(p, v0 + lane);
        if (lane == 0) {
            mbar_wait(&empty[p_stage], p_phase ^ 1);
            mbar_expect_tx(&full[p_stage], (uint32_t)(rows * cols4 * 16));
        }
        __syncwarp();
        if (lane < rows)
            tma_load_1d(ring + (size_t)p_stage * TMA_STAGE_FLOATS + lane * NT * 4, p_row + (size_t)c0 * 4,
                        (uint32_t)(cols4 * 16), &full[p_stage]);
        ++p_it;
        if (++p_step == nsteps) { p_step = 0; ++p_tile; }
        if (++p_stage == NSTAGE) { p_stage = 0; p_phase ^= 1; }
    };
    if (warp == NWARP) {
        // ---- producer warp.  It runs on its own: issuing one stage costs ~0.5 us (8 bulk copies), so
        // the other warps must not meet it at a barrier (measured r02: with the producer inside the
        // prologue's barriers the activation vector was staged 5.3 us after the dependency wait, and
        // the memory pipe sat idle behind a full ring).
        // Only nprefill stages go out before the wait: the activation vector's bulk copy is issued by
        // warp 0 right after the wait and is served behind everything this SM already requested
        // (~47 GB/s of HBM per SM: a full 192 KB ring ahead of it costs 4 us).
        while (p_it < total && p_it < p.nprefill) produce_one();
        if (p_it >= total) pdl_launch_dependents();
        if (lane == 0) L2B_STAMP(p.trace, 1);
        pdl_wait();
        if (!p.ctl[CTL_DONE]) {
            while (p_it < total) {
                produce_one();
                if (p_it == total) pdl_launch_dependents();   // last stage in flight
            }
            if (lane == 0) L2B_STAMP(p.trace, 6);
            return;
        }
    }

    // the rmsnorm gain is immutable: fetch this thread's slice before waiting on the previous
    // kernel (on big models it has been evicted from L2 by the weight stream, and after the wait
    // its DRAM round trip would queue behind this CTA's own ring traffic)
    constexpr int MAXV = 5;                               // n <= 5 * 288 * 4 = 5760 floats when fused
    constexpr int PRO_THREADS = TMA_THREADS - 32;         // consumers + epilogue warp
    const int ptid = tid < NT ? tid : tid - 32;           // index among the prologue's threads
    float4 gv[MAXV];
    if (p.gamma && warp != NWARP) {
        const float4 *g4 = reinterpret_cast<const float4 *>(p.gamma);
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = ptid + k * PRO_THREADS;
            gv[k] = (i < n4) ? __ldg(g4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }

    // ---- everything below reads what earlier kernels of this step wrote
    if (warp != NWARP) pdl_wait();
    if (p.ctl[CTL_DONE]) {
        // generation already ended: drain the bulk copies already aimed at our shared memory
        if (tid == 0)
            for (int s = 0; s < p.nprefill && s < total; ++s) mbar_wait(&full[s], 0);
        __syncthreads();
        return;
    }
    const int pos = p.ctl[CTL_POS];
    if (p.bump_epoch && blockIdx.x == 0 && tid == 0) const_cast<int *>(p.ctl)[CTL_EPOCH] += 1;
    if (tid == 0) L2B_STAMP(p.trace, 2);

    // stage the activation vector (consumer warps + epilogue warp; barrier 1 is theirs)
    {
        const float *xsrc = p.emb ? p.emb + (size_t)p.ctl[CTL_TOKEN] * p.n : p.x_in;
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)p.n * 4u;
            mbar_expect_tx(&xbar, bytes);
            tma_load_1d(xs, xsrc, bytes, &xbar);
        }
        // epilogue warp: this position's RoPE row.  The table row comes from DRAM on big models (the
        // weight stream evicts it), so it is only FETCHED here, into registers; it is parked in shared
        // memory after the prologue's last barrier — the other warps must not wait for it
        // (measured r02: it held the qkv prologue 1.4 us longer than the w13 one)
        float rc_reg[4], rs_reg[4];
        if (EPI == EPI_QKV && tid >= NT + 32) {
            const int half = p.head_size >> 1;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = lane + 32 * k;
                rc_reg[k] = (i < half) ? __ldg(p.rope_cos + (size_t)pos * half + i) : 0.0f;
                rs_reg[k] = (i < half) ? __ldg(p.rope_sin + (size_t)pos * half + i) : 0.0f;
            }
        }
        mbar_wait(&xbar, 0);
        if (p.gamma || p.x_out) {
            float4 *xs4w = reinterpret_cast<float4 *>(xs);
            float ssq = 0.0f;
#pragma unroll
            for (int k = 0; k < MAXV; ++k) {
                const int i = ptid + k * PRO_THREADS;
                if (i < n4) {
                    const float4 v = xs4w[i];
                    if (p.x_out && blockIdx.x == 0) reinterpret_cast<float4 *>(p.x_out)[i] = v;
                    ssq = fmaf(v.x, v.x, ssq); ssq = fmaf(v.y, v.y, ssq);
                    ssq = fmaf(v.z, v.z, ssq); ssq = fmaf(v.w, v.w, ssq);
                }
            }
            if (p.gamma) {
                ssq = warp_sum(ssq);
                if (lane == 0) scratch[ptid >> 5] = ssq;
                named_bar_sync(1, PRO_THREADS);
                float ss = (lane < PRO_THREADS / 32) ? scratch[lane] : 0.0f;
                ss = warp_sum(ss);
                ss /= (float)p.n;            // :452
                ss += 1e-5f;                 // :453
                const float sc = 1.0f / sqrtf(ss);  // :454
#pragma unroll
                for (int k = 0; k < MAXV; ++k) {
                    const int i = ptid + k * PRO_THREADS;
                    if (i < n4) {
                        float4 v = xs4w[i];
                        v.x = __fmul_rn(__fmul_rn(v.x, sc), gv[k].x);   // (x*s)*w, :462
                        v.y = __fmul_rn(__fmul_rn(v.y, sc), gv[k].y);
                        v.z = __fmul_rn(__fmul_rn(v.z, sc), gv[k].z);
                        v.w = __fmul_rn(__fmul_rn(v.w, sc), gv[k].w);
                        xs4w[i] = v;
                    }
                }
            }
        }
        named_bar_sync(1, PRO_THREADS);
        if (EPI == EPI_QKV && tid >= NT + 32) {
            const int half = p.head_size >> 1;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = lane + 32 * k;
                if (i < half) { rope_s[0][i] = rc_reg[k]; rope_s[1][i] = rs_reg[k]; }
            }
            __syncwarp();
        }
    }
    if (tid == 0) L2B_STAMP(p.trace, 3);

    if (warp == NWARP + 1) {
        // ---- epilogue warp: lanes 0..3 own the four row pairs of each tile
        unsigned long long best = 0ull;
        const unsigned int epoch = (EPI == EPI_XCHG) ? (unsigned int)p.ctl[CTL_EPOCH] : 0u;
        // EPI_RESID: the residual values of tile t+1 are fetched while tile t is being reduced
        float2 xr_next = gemv_resid_fetch<EPI>(p, (lane < GEMV8_R / 2 && r0 + 2 * lane < r1) ? r0 + 2 * lane : p.total_rows);
        for (int t = 0; t < ntiles; ++t) {
            const int par = t & 1, use = t >> 1;
            const float2 xr = xr_next;
            {
                const int vn = r0 + (t + 1) * GEMV8_R + 2 * lane;
                xr_next = gemv_resid_fetch<EPI>(p, (lane < GEMV8_R / 2 && vn < r1) ? vn : p.total_rows);
            }
            mbar_wait(&tile_full[par], use & 1);
            float s0 = 0.0f, s1 = 0.0f;
            if (lane < GEMV8_R / 2) {
#pragma unroll
                for (int w8 = 0; w8 < NWARP; ++w8) {       // fixed order
                    s0 += red[par][w8][2 * lane];
                    s1 += red[par][w8][2 * lane + 1];
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&tile_free[par]);  // consumers may overwrite red[par]
            const int vp = r0 + t * GEMV8_R + 2 * lane;
            if (lane < GEMV8_R / 2 && vp < r1) {
                if (EPI == EPI_QKV && vp < p.rows0 + p.rows1) {
                    const bool is_q = vp < p.rows0;
                    const int i = is_q ? vp : vp - p.rows0;
                    const int pr = (i % p.head_size) >> 1;                                  // :338
                    const float fcr = rope_s[0][pr], fci = rope_s[1][pr];
                    const float q0 = __fsub_rn(__fmul_rn(s0, fcr), __fmul_rn(s1, fci));      // :348
                    const float q1 = __fadd_rn(__fmul_rn(s0, fci), __fmul_rn(s1, fcr));      // :349
                    float *dst = is_q ? p.out0 + i : p.kcache + (size_t)pos * p.kv_dim + i;  // :355,:357
                    *reinterpret_cast<float2 *>(dst) = make_float2(q0, q1);
                } else {
                    gemv_epilogue_pair<EPI>(p, vp, s0, s1, pos, best, epoch, xr);
                }
            }
        }
        if (EPI == EPI_ARGMAX) {
#pragma unroll
            for (int o = 2; o > 0; o >>= 1) {
                const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
                best = other > best ? other : best;
            }
            if (lane == 0 && best) atomicMax(p.amax, best);
        }
        if (EPI == EPI_XCHG && p.xres) tp_reduce_tail(p, epoch, lane);
        if (lane == 0) L2B_STAMP(p.trace, 7);
        return;
    }

    // ---- consumers (warps 0..7)
    const float4 *xs4 = reinterpret_cast<const float4 *>(xs);
    float acc[GEMV8_R];
#pragma unroll
    for (int r = 0; r < GEMV8_R; ++r) acc[r] = 0.0f;
    int c_stage = 0;
    uint32_t c_phase = 0;
    int t = 0, st = 0;
    for (int it = 0; it < total; ++it, ++st) {
        if (st == nsteps) { st = 0; ++t; }
        const int c = st * NT + tid;
        const int v0 = r0 + t * GEMV8_R;
        const int rows = min(GEMV8_R, r1 - v0);
        mbar_wait(&full[c_stage], c_phase);
        if (it == 0 && tid == 0) L2B_STAMP(p.trace, 4);
        if (c < n4) {
            const float4 *w4 = reinterpret_cast<const float4 *>(ring + (size_t)c_stage * TMA_STAGE_FLOATS) + tid;
            const float4 xv = xs4[c];
#pragma unroll
            for (int r = 0; r < GEMV8_R; ++r)
                if (r < rows) acc[r] = dot4(w4[r * NT], xv, acc[r]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[c_stage]);      // this warp is done with the stage
        if (++c_stage == NSTAGE) { c_stage = 0; c_phase ^= 1; }
        if (it == total - 1 && tid == 0) L2B_STAMP(p.trace, 5);
        if (st != nsteps - 1) continue;
        // ---- end of a tile: transposing butterfly, lane L (L % 4 == 0) ends with row L / 4
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float send = (lane & 16) ? acc[i] : acc[i + 4];
            const float keep = (lane & 16) ? acc[i + 4] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float send = (lane & 8) ? acc[i] : acc[i + 2];
            const float keep = (lane & 8) ? acc[i + 2] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {
            const float send = (lane & 4) ? acc[0] : acc[1];
            const float keep = (lane & 4) ? acc[1] : acc[0];
            acc[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 2);
        acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
        const int par = t & 1, use = t >> 1;
        mbar_wait(&tile_free[par], (use & 1) ^ 1);        // epilogue warp has read use-1 of red[par]
        if ((lane & 3) == 0) red[par][warp][lane >> 2] = acc[0];
        __syncwarp();
        if (lane == 0) mbar_arrive(&tile_full[par]);
#pragma unroll
        for (int r = 0; r < GEMV8_R; ++r) acc[r] = 0.0f;
    }
}

// Scalar fallback for shapes the vector kernel cannot take (n % 4 != 0 or unaligned rows):
// one warp per row.  Only reachable from l2b_op_matmul (the reference KATs use n = 3, 12).
__global__ void __launch_bounds__(NT) gemv_scalar_kernel(float *out, const float *x, const float *w,
                                                         int d, int n) {
    const int warp = (blockIdx.x * NT + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * NT) >> 5;
    for (int row = warp; row < d; row += nwarps) {
        float acc = 0.0f;
        for (int c = lane; c < n; c += 32) acc = fmaf(w[(size_t)row * n + c], x[c], acc);
        acc = warp_sum(acc);
        if (lane == 0) out[row] = acc;
    }
}

// ---------------------------------------------------------------------------------------
// Per-head attention over the KV cache (src/main.zig:361-389), split along the timeline.
//
// grid = (n_heads, nsplit).  CTA (h, s) owns positions [s*chunk, min((s+1)*chunk, pos+1)):
//   scores = q_h . K[t] / sqrt(head_size)   (:367-375)  -> shared memory
//   softmax pieces: max, exp, sum           (:687-706)
//   out = sum_t p[t] * V[t]                 (:657-685)
// With one active split the normalised weights are formed first (x/sum, :703-705) exactly as
// the reference does; with several, partial (max, sum, unnormalised out) triples are merged
// by the last CTA of the head to arrive (threadfence + counter), in fixed split order, so the
// result is deterministic.
// ---------------------------------------------------------------------------------------
// One activation vector of a batched pass (prompt prefill, or decode streams that share one copy of
// the weights): its own token, position and KV cache.  Prefill fills consecutive positions of one
// cache; batched decode has one entry per stream.  Device memory, so a step reads it the way a
// single-stream step reads ctl, and advance_batch_kernel moves it on without the host.
struct BatchVec {
    int token, pos;
    int done;              // this vector's generation ended: every later kernel skips it (no KV append)
    int step, limit;       // generate loop: steps taken, steps allowed
    int pad;
    float *kc, *vc;        // this vector's (n_layers, seq_len, kv_dim) key / value caches
};

struct AttnParams {
    const int *ctl;
    const float *q;        // (n_heads * head_size)
    const float *kcache;   // this layer: (seq_len, kv_dim)
    const float *vcache;
    float *xb;             // (n_heads * head_size)
    float *part_o;         // (n_heads, nsplit, head_size)
    float *part_ml;        // (n_heads, nsplit, 2)
    unsigned int *counters;  // (n_heads), zero between launches
    int head_size, kv_dim, kv_mul, nsplit, min_chunk;
    unsigned long long *trace;
    // batched passes: gridDim.z queries at once; query z takes its position, cache (vec[z].kc/vc +
    // kv_off) and done flag from vec[z] and uses q / xb / partial buffers offset by z (vec == nullptr:
    // single position from the control block, cache kcache / vcache)
    const BatchVec *vec;
    size_t kv_off;
    int q_stride;
    int seq_len;           // rows of the cache (bounds the speculative first pass; 0 = no speculation)
};

__device__ __forceinline__ int attn_lanes_per_row(int hs4) {
    return (hs4 % 8 == 0) ? 8 : (hs4 % 4 == 0) ? 4 : (hs4 % 2 == 0) ? 2 : 1;
}

// scores for positions [t0,t1) of one head into sc[0..t1-t0); q fragments live in registers
__device__ __forceinline__ void attn_scores(float *sc, const float *qg, const float *kbase,
                                            int kv_dim, int head_size, int t0, int t1) {
    const int hs4 = head_size >> 2;
    const int lpr = attn_lanes_per_row(hs4);
    const int nf = hs4 / lpr;
    const int rows_per_warp = 32 / lpr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lr = lane % lpr, rw = lane / lpr;
    const float4 *q4 = reinterpret_cast<const float4 *>(qg);
    const float root_hs = sqrtf((float)head_size);
    for (int tb = t0 + warp * rows_per_warp; tb < t1; tb += NWARP * rows_per_warp) {
        const int t = tb + rw;
        float acc = 0.0f;
        if (t < t1) {
            const float4 *k4 = reinterpret_cast<const float4 *>(kbase + (size_t)t * kv_dim);
            for (int f = 0; f < nf; ++f) {
                const int j = lr + f * lpr;
                acc = dot4(__ldg(k4 + j), __ldg(q4 + j), acc);
            }
        }
        for (int o = lpr >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (t < t1 && lr == 0) sc[t - t0] = acc / root_hs;   // score /= sqrt(head_size), :372
    }
}

// red[g][0..head_size) = sum over this group's rows of w[t-t0] * V[t]   (G = NT / (head_size/4))
__device__ __forceinline__ void attn_weighted_rows(float *red, const float *w, const float *vbase,
                                                   int kv_dim, int head_size, int t0, int t1) {
    const int hs4 = head_size >> 2;
    const int G = NT / hs4;
    const int tid = threadIdx.x;
    const int g = tid / hs4, c = tid % hs4;
    if (g < G) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int t = t0 + g; t < t1; t += G) {
            const float wt = w[t - t0];
            const float4 v = __ldg(reinterpret_cast<const float4 *>(vbase + (size_t)t * kv_dim) + c);
            a.x = fmaf(v.x, wt, a.x); a.y = fmaf(v.y, wt, a.y);
            a.z = fmaf(v.z, wt, a.z); a.w = fmaf(v.w, wt, a.w);
        }
        reinterpret_cast<float4 *>(red)[g * hs4 + c] = a;
    }
}

__global__ void __launch_bounds__(NT) attention_kernel(const AttnParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int is_last;
    unsigned long long *atr = p.trace ? p.trace + ((size_t)blockIdx.y * gridDim.x) * TRACE_SLOTS : nullptr;
    if (threadIdx.x == 0) L2B_STAMP(atr, 0);
    pdl_launch_dependents();
    pdl_wait();
    if (threadIdx.x == 0) L2B_STAMP(atr, 2);
    if (p.ctl[CTL_DONE]) return;

    const int h = blockIdx.x, s = blockIdx.y;
    const int hs = p.head_size;
    const int T = p.ctl[CTL_POS] + 1;
    int chunk = (T + p.nsplit - 1) / p.nsplit;
    if (chunk < p.min_chunk) chunk = p.min_chunk;
    const int active = (T + chunk - 1) / chunk;
    if (s >= active) return;
    const int t0 = s * chunk;
    const int t1 = min(T, t0 + chunk);
    const int len = t1 - t0;

    // shared layout: red[G*hs] | sc[chunk_cap]
    const int hs4 = hs >> 2;
    const int G = NT / hs4;
    float *red = reinterpret_cast<float *>(smem_raw);
    float *sc = red + G * hs;

    const int tid = threadIdx.x, lane = tid & 31;
    const size_t hoff = (size_t)(h / p.kv_mul) * hs;   // :369, :382

    attn_scores(sc, p.q + (size_t)h * hs, p.kcache + hoff, p.kv_dim, hs, t0, t1);
    __syncthreads();

    // softmax pieces (:690-705).  Every warp recomputes max and sum over the whole split from
    // shared memory (identical order in every warp), which costs a few shuffles instead of
    // four block-wide barriers.
    float m = -INFINITY;
    for (int i = lane; i < len; i += 32) m = fmaxf(m, sc[i]);
    m = warp_max(m);
    __syncthreads();   // every warp has read the raw scores before anyone overwrites them
    for (int i = tid; i < len; i += NT) sc[i] = expf(sc[i] - m);   // :699
    __syncthreads();
    float l = 0.0f;
    for (int i = lane; i < len; i += 32) l += sc[i];
    l = warp_sum(l);

    attn_weighted_rows(red, sc, p.vcache + hoff, p.kv_dim, hs, t0, t1);
    __syncthreads();
    float o = 0.0f;
    if (tid < hs) {
        for (int gg = 0; gg < G; ++gg) o += red[gg * hs + tid];   // fixed order
    }

    if (active == 1) {
        if (tid < hs) p.xb[(size_t)h * hs + tid] = o / l;        // normalisation of :703-705
        if (tid == 0) L2B_STAMP(atr, 7);
        return;
    }

    // ---- publish the partial, last arriver merges
    if (tid < hs) p.part_o[((size_t)h * p.nsplit + s) * hs + tid] = o;
    if (tid == 0) {
        p.part_ml[((size_t)h * p.nsplit + s) * 2 + 0] = m;
        p.part_ml[((size_t)h * p.nsplit + s) * 2 + 1] = l;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned int prev = atomicAdd(&p.counters[h], 1u);
        is_last = (prev == (unsigned int)(active - 1));
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (tid == 0) p.counters[h] = 0u;  // ready for the next launch
    const volatile float *ml = p.part_ml + (size_t)h * p.nsplit * 2;
    float M = -INFINITY;
    for (int j = 0; j < active; ++j) M = fmaxf(M, ml[j * 2]);
    float Lsum = 0.0f;
    for (int j = 0; j < active; ++j) Lsum += expf(ml[j * 2] - M) * ml[j * 2 + 1];
    if (tid < hs) {
        const volatile float *pb = p.part_o + (size_t)h * p.nsplit * hs;
        float acc = 0.0f;
        for (int j = 0; j < active; ++j) acc = fmaf(expf(ml[j * 2] - M), pb[(size_t)j * hs + tid], acc);
        p.xb[(size_t)h * hs + tid] = acc / Lsum;
    }
}

// ---------------------------------------------------------------------------------------
// attention, flash-decoding form (default).  The three-pass kernel above has a long dependent
// chain (scores -> barrier -> max -> barrier -> exp -> barrier -> sum -> V pass -> barrier ->
// fold; 9.7 us per layer at pos 40 on llama2-7B, profiles/r01_trace_7b.txt).  Here every group
// of LPR lanes owns whole timeline rows and keeps a running (max, sum, weighted V slice) in
// registers, with the K and V loads of two rows in flight together, so the only barriers are the
// two around the final merge of the 8 * (32/LPR) groups in shared memory.
//   score_t = q . K_t / sqrt(hs)                                   (:367-375)
//   online softmax: m' = max(m, s); l = l*e^(m-m') + e^(s-m'); acc = acc*e^(m-m') + e^(s-m') V_t
//   out = sum_groups e^(m_g-M) acc_g / sum_groups e^(m_g-M) l_g    (== softmax(:687-706) . V, :657-685)
// ---------------------------------------------------------------------------------------
// Merge the online-softmax partials (m, l, acc) of the RPW row groups of ONE warp with xor shuffles
// (lanes with equal column slice `lr`, different row group): log2(RPW) steps in a fixed tree order,
// so only NWARP partials per CTA go through shared memory afterwards.  Measured r02 (cluster-kernel
// phase trace): the previous all-groups-through-shared-memory merge (64 groups, then a 64-term serial
// sum per output element) was 1.8 us of a 2.4 us attention.
template <int NF>
__device__ __forceinline__ void attn_warp_merge(float &m, float &l, float4 (&acc)[NF], int LPR) {
    for (int off = LPR; off < 32; off <<= 1) {
        const float mo = __shfl_xor_sync(0xffffffffu, m, off);
        const float lo = __shfl_xor_sync(0xffffffffu, l, off);
        const float mn = fmaxf(m, mo);
        const float ss = (m == -INFINITY) ? 0.0f : expf(m - mn);     // empty partials carry m = -inf, l = 0
        const float so = (mo == -INFINITY) ? 0.0f : expf(mo - mn);
        l = fmaf(l, ss, lo * so);
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            const float ox = __shfl_xor_sync(0xffffffffu, acc[f].x, off);
            const float oy = __shfl_xor_sync(0xffffffffu, acc[f].y, off);
            const float oz = __shfl_xor_sync(0xffffffffu, acc[f].z, off);
            const float ow = __shfl_xor_sync(0xffffffffu, acc[f].w, off);
            acc[f].x = fmaf(acc[f].x, ss, ox * so);
            acc[f].y = fmaf(acc[f].y, ss, oy * so);
            acc[f].z = fmaf(acc[f].z, ss, oz * so);
            acc[f].w = fmaf(acc[f].w, ss, ow * so);
        }
        m = mn;
    }
}

template <int NF>   // float4 per lane per row: head_size = 4 * NF * LPR
__global__ void __launch_bounds__(NT) attention_flash_kernel(const AttnParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int is_last;
    unsigned long long *atr = p.trace ? p.trace + ((size_t)blockIdx.y * gridDim.x) * TRACE_SLOTS : nullptr;
    if (threadIdx.x == 0) L2B_STAMP(atr, 0);
    pdl_launch_dependents();
    pdl_wait();
    if (threadIdx.x == 0) L2B_STAMP(atr, 2);

    const int h = blockIdx.x, s = blockIdx.y, z = blockIdx.z;
    const int hs = p.head_size, hs4 = hs >> 2;
    const int LPR = hs4 / NF;                 // lanes per row (8, 4, 2 or 1)
    const int RPW = 32 / LPR;                 // rows per warp pass
    const int NG = NWARP * RPW;               // row groups in the CTA
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lr = lane % LPR, rw = lane / LPR;
    const float *qz = p.q + (size_t)z * p.q_stride;
    const size_t hoff = (size_t)(h / p.kv_mul) * hs;          // :369, :382
    const float4 *q4 = reinterpret_cast<const float4 *>(qz + (size_t)h * hs);
    const float *kb = (p.vec ? p.vec[z].kc + p.kv_off : p.kcache) + hoff;
    const float *vb = (p.vec ? p.vec[z].vc + p.kv_off : p.vcache) + hoff;

    // Everything whose ADDRESS does not depend on the position is requested before the position is
    // read from the control block: q, and (timeline split 0) the cache rows of this lane's first pass —
    // rows beyond pos hold stale data and are masked below.  One L2 round trip less on the chain
    // control word -> rows -> softmax (measured r02: attention is 2.7 us of a 13 us stories15M layer).
    float4 qf[NF], acc[NF], ka[NF], vA[NF], kc[NF], vC[NF];
    const int ta0 = warp * RPW + rw, tc0 = ta0 + NG;
    const bool spec = (s == 0) && tc0 < p.seq_len;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
        qf[f] = __ldcg(q4 + lr + f * LPR);
        acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (spec) {
        const float4 *ka4 = reinterpret_cast<const float4 *>(kb + (size_t)ta0 * p.kv_dim);
        const float4 *va4 = reinterpret_cast<const float4 *>(vb + (size_t)ta0 * p.kv_dim);
        const float4 *kc4 = reinterpret_cast<const float4 *>(kb + (size_t)tc0 * p.kv_dim);
        const float4 *vc4 = reinterpret_cast<const float4 *>(vb + (size_t)tc0 * p.kv_dim);
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            ka[f] = __ldcg(ka4 + lr + f * LPR);
            vA[f] = __ldcg(va4 + lr + f * LPR);
            kc[f] = __ldcg(kc4 + lr + f * LPR);
            vC[f] = __ldcg(vc4 + lr + f * LPR);
        }
    }

    if (p.vec ? p.vec[z].done : p.ctl[CTL_DONE]) return;
    const int T = (p.vec ? p.vec[z].pos : p.ctl[CTL_POS]) + 1;
    int chunk = (T + p.nsplit - 1) / p.nsplit;
    if (chunk < p.min_chunk) chunk = p.min_chunk;
    const int active = (T + chunk - 1) / chunk;
    if (s >= active) return;
    const int t0 = s * chunk;
    const int t1 = min(T, t0 + chunk);
    float *xbz = p.xb + (size_t)z * p.q_stride;
    float *part_o_z = p.part_o + (size_t)z * gridDim.x * p.nsplit * hs;
    float *part_ml_z = p.part_ml + (size_t)z * gridDim.x * p.nsplit * 2;
    unsigned int *counters_z = p.counters + (size_t)z * gridDim.x;
    float *accp = reinterpret_cast<float *>(smem_raw);        // [NG][hs]
    float *mlp = accp + (size_t)NG * hs;                      // [NG][2]
    const float root_hs = sqrtf((float)hs);
    float m = -INFINITY, l = 0.0f;

    auto update = [&](const float4 (&kv)[NF], const float4 (&vv)[NF], bool valid) {
        float sc = 0.0f;
#pragma unroll
        for (int f = 0; f < NF; ++f) sc = dot4(kv[f], qf[f], sc);
        for (int o = LPR >> 1; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
        if (!valid) return;
        sc = sc / root_hs;                                    // :372
        const float mn = fmaxf(m, sc);
        const float scale = expf(m - mn);                     // 0 on the first row (m = -inf)
        const float pw = expf(sc - mn);
        l = fmaf(l, scale, pw);
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            acc[f].x = fmaf(acc[f].x, scale, pw * vv[f].x);
            acc[f].y = fmaf(acc[f].y, scale, pw * vv[f].y);
            acc[f].z = fmaf(acc[f].z, scale, pw * vv[f].z);
            acc[f].w = fmaf(acc[f].w, scale, pw * vv[f].w);
        }
        m = mn;
    };

    // two rows per pass: 4*NF 128-bit loads in flight per lane before any arithmetic
    // NOTE: the loop bound is warp-uniform (row groups of one warp must run the same number of
    // passes: `update` contains full-mask shuffles); per-lane validity is handled inside.
    for (int tbw = t0 + warp * RPW; tbw < t1; tbw += 2 * NG) {
        const int ta = tbw + rw, tc = ta + NG;
        const bool va = ta < t1, vc = tc < t1;
        if (!(spec && tbw == warp * RPW)) {                   // the first pass of split 0 is already in registers
            const float4 *ka4 = reinterpret_cast<const float4 *>(kb + (size_t)(va ? ta : t0) * p.kv_dim);
            const float4 *va4 = reinterpret_cast<const float4 *>(vb + (size_t)(va ? ta : t0) * p.kv_dim);
            const float4 *kc4 = reinterpret_cast<const float4 *>(kb + (size_t)(vc ? tc : t0) * p.kv_dim);
            const float4 *vc4 = reinterpret_cast<const float4 *>(vb + (size_t)(vc ? tc : t0) * p.kv_dim);
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                ka[f] = __ldcg(ka4 + lr + f * LPR);
                vA[f] = __ldcg(va4 + lr + f * LPR);
                kc[f] = __ldcg(kc4 + lr + f * LPR);
                vC[f] = __ldcg(vc4 + lr + f * LPR);
            }
        }
        update(ka, vA, va);
        update(kc, vC, vc);
    }

    // ---- merge: row groups of a warp by shuffles, then the NWARP warps through shared memory (fixed
    // order => deterministic)
    attn_warp_merge<NF>(m, l, acc, LPR);
    if (rw == 0) {
#pragma unroll
        for (int f = 0; f < NF; ++f)
            reinterpret_cast<float4 *>(accp + (size_t)warp * hs)[lr + f * LPR] = acc[f];
        if (lr == 0) { mlp[2 * warp] = m; mlp[2 * warp + 1] = l; }
    }
    __syncthreads();
    float M = -INFINITY;
#pragma unroll
    for (int g = 0; g < NWARP; ++g) M = fmaxf(M, mlp[2 * g]);
    float L = 0.0f, o = 0.0f;
#pragma unroll
    for (int g = 0; g < NWARP; ++g) {                          // every thread: same order, same values
        const float w = (mlp[2 * g] == -INFINITY) ? 0.0f : expf(mlp[2 * g] - M);
        L = fmaf(w, mlp[2 * g + 1], L);
        if (tid < hs) o = fmaf(w, accp[(size_t)g * hs + tid], o);
    }

    if (active == 1) {
        if (tid < hs) xbz[(size_t)h * hs + tid] = o / L;
        if (tid == 0) L2B_STAMP(atr, 7);
        return;
    }

    // ---- several timeline splits: publish (M, L, unnormalised out), last arriver merges
    if (tid < hs) part_o_z[((size_t)h * p.nsplit + s) * hs + tid] = o;
    if (tid == 0) {
        part_ml_z[((size_t)h * p.nsplit + s) * 2 + 0] = M;
        part_ml_z[((size_t)h * p.nsplit + s) * 2 + 1] = L;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned int prev = atomicAdd(&counters_z[h], 1u);
        is_last = (prev == (unsigned int)(active - 1));
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (tid == 0) counters_z[h] = 0u;  // ready for the next launch
    const volatile float *ml = part_ml_z + (size_t)h * p.nsplit * 2;
    float MM = -INFINITY;
    for (int j = 0; j < active; ++j) MM = fmaxf(MM, ml[j * 2]);
    float Lsum = 0.0f;
    for (int j = 0; j < active; ++j) Lsum += expf(ml[j * 2] - MM) * ml[j * 2 + 1];
    if (tid < hs) {
        const volatile float *pb = part_o_z + (size_t)h * p.nsplit * hs;
        float a2 = 0.0f;
        for (int j = 0; j < active; ++j) a2 = fmaf(expf(ml[j * 2] - MM), pb[(size_t)j * hs + tid], a2);
        xbz[(size_t)h * hs + tid] = a2 / Lsum;
    }
}

// ---------------------------------------------------------------------------------------
// Small models (stories15M / 110M): a decode step there is a chain of ~3 us kernels that move
// <= 2 MB each, so the step time is the NUMBER of kernels.  One fusion survived measurement
// (profiles/r02_small_models.md; the fused-FFN kernel and the all-layers cluster kernel that were
// also built are parked in scripts/experiments/):
//
// attn_wo_kernel: attention of one head (:361-389) + that head's column slice of wo (:392) in one
//   thread-block CLUSTER of R CTAs.  CTA s of the cluster runs flash-decoding over timeline split s;
//   the R partial (max, sum, unnormalised out) triples are merged through DISTRIBUTED SHARED MEMORY
//   (every CTA reads its peers' triples after a cluster barrier, in fixed split order), then CTA s
//   multiplies the merged head output with rows [s*dim/R, (s+1)*dim/R) of wo[:, h*hs:(h+1)*hs] and
//   writes parts[h][row].  The consumer's prologue completes the product: x += sum_h parts[h]
//   (fixed head order), which is the wo GEMV's own summation split at head boundaries.
// ---------------------------------------------------------------------------------------
struct AttnWoParams {
    AttnParams a;
    const float *wo;        // this layer's (dim, q_dim) row-major
    float *parts;           // (n_heads, dim)
    int dim, q_dim;
};

template <int NF>   // float4 per lane per row: head_size = 4 * NF * LPR
__global__ void __launch_bounds__(NT) attn_wo_kernel(const AttnWoParams q) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const AttnParams &p = q.a;
    const int h = blockIdx.x, s = blockIdx.y, R = gridDim.y;     // cluster = the R CTAs of one head
    const int hs = p.head_size, hs4 = hs >> 2;
    const int LPR = hs4 / NF, RPW = 32 / LPR, NG = NWARP * RPW;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lr = lane % LPR, rw = lane / LPR;
    float *accp = reinterpret_cast<float *>(smem_raw);        // [NG][hs]
    float *mlp = accp + (size_t)NG * hs;                      // [NG][2]
    float *wgt = mlp + 2 * NG;                                // [NG]
    float *tri = wgt + NG;                                    // [hs + 4]: this CTA's unnormalised out, M, L
    float *xbs = tri + hs + 4;                                // [hs]: merged head output

    // rows of the wo slice this CTA produces; the first pass of weights is immutable: fetch it now
    const int rows_per = (q.dim + R - 1) / R;
    const int r0 = s * rows_per, r1 = min(q.dim, r0 + rows_per);
    const float4 *wo4 = reinterpret_cast<const float4 *>(q.wo) + (size_t)h * hs4;
    const int q4 = q.q_dim >> 2;
    float4 wpre[NF];
    {
        const int row = r0 + warp * RPW + rw;
#pragma unroll
        for (int f = 0; f < NF; ++f)
            wpre[f] = (row < r1) ? ldg_stream(wo4 + (size_t)row * q4 + lr + f * LPR) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    pdl_launch_dependents();
    pdl_wait();
    if (p.ctl[CTL_DONE]) return;                               // uniform over the whole grid

    const int T = p.ctl[CTL_POS] + 1;
    const int chunk = (T + R - 1) / R;
    const int t0 = s * chunk, t1 = min(T, t0 + chunk);         // may be empty (t0 >= T)
    const size_t hoff = (size_t)(h / p.kv_mul) * hs;           // :369, :382
    const float4 *qv4 = reinterpret_cast<const float4 *>(p.q + (size_t)h * hs);
    const float *kb = p.kcache + hoff, *vb = p.vcache + hoff;
    const float root_hs = sqrtf((float)hs);

    float4 qf[NF], acc[NF];
#pragma unroll
    for (int f = 0; f < NF; ++f) {
        qf[f] = __ldcg(qv4 + lr + f * LPR);
        acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float m = -INFINITY, l = 0.0f;
    auto update = [&](const float4 (&kv)[NF], const float4 (&vv)[NF], bool valid) {
        float sc = 0.0f;
#pragma unroll
        for (int f = 0; f < NF; ++f) sc = dot4(kv[f], qf[f], sc);
        for (int o = LPR >> 1; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
        if (!valid) return;
        sc = sc / root_hs;                                    // :372
        const float mn = fmaxf(m, sc);
        const float scale = expf(m - mn);
        const float pw = expf(sc - mn);
        l = fmaf(l, scale, pw);
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            acc[f].x = fmaf(acc[f].x, scale, pw * vv[f].x);
            acc[f].y = fmaf(acc[f].y, scale, pw * vv[f].y);
            acc[f].z = fmaf(acc[f].z, scale, pw * vv[f].z);
            acc[f].w = fmaf(acc[f].w, scale, pw * vv[f].w);
        }
        m = mn;
    };
    for (int tbw = t0 + warp * RPW; tbw < t1; tbw += 2 * NG) {   // warp-uniform bound (full-mask shuffles inside)
        const int ta = tbw + rw, tc = ta + NG;
        const bool va = ta < t1, vc = tc < t1;
        float4 ka[NF], vA[NF], kc[NF], vC[NF];
        const float4 *ka4 = reinterpret_cast<const float4 *>(kb + (size_t)(va ? ta : t0) * p.kv_dim);
        const float4 *va4 = reinterpret_cast<const float4 *>(vb + (size_t)(va ? ta : t0) * p.kv_dim);
        const float4 *kc4 = reinterpret_cast<const float4 *>(kb + (size_t)(vc ? tc : t0) * p.kv_dim);
        const float4 *vc4 = reinterpret_cast<const float4 *>(vb + (size_t)(vc ? tc : t0) * p.kv_dim);
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            ka[f] = __ldcg(ka4 + lr + f * LPR);
            vA[f] = __ldcg(va4 + lr + f * LPR);
            kc[f] = __ldcg(kc4 + lr + f * LPR);
            vC[f] = __ldcg(vc4 + lr + f * LPR);
        }
        update(ka, vA, va);
        update(kc, vC, vc);
    }
    // ---- merge: row groups of a warp by shuffles, then the NWARP warps through shared memory
    attn_warp_merge<NF>(m, l, acc, LPR);
    if (rw == 0) {
#pragma unroll
        for (int f = 0; f < NF; ++f)
            reinterpret_cast<float4 *>(accp + (size_t)warp * hs)[lr + f * LPR] = acc[f];
        if (lr == 0) { mlp[2 * warp] = m; mlp[2 * warp + 1] = l; }
    }
    __syncthreads();
    {
        float M = -INFINITY;
#pragma unroll
        for (int g = 0; g < NWARP; ++g) M = fmaxf(M, mlp[2 * g]);
        float L = 0.0f, o = 0.0f;
#pragma unroll
        for (int g = 0; g < NWARP; ++g) {
            const float w = (mlp[2 * g] == -INFINITY) ? 0.0f : expf(mlp[2 * g] - M);
            L = fmaf(w, mlp[2 * g + 1], L);
            if (tid < hs) o = fmaf(w, accp[(size_t)g * hs + tid], o);
        }
        if (tid < hs) tri[tid] = o;
        if (tid == 0) { tri[hs] = M; tri[hs + 1] = L; }
    }
    // ---- merge the R timeline splits of the head through distributed shared memory
    cluster.sync();
    {
        float MM = -INFINITY;
        for (int j = 0; j < R; ++j) MM = fmaxf(MM, cluster.map_shared_rank(tri, j)[hs]);
        float Lsum = 0.0f, a2 = 0.0f;
        for (int j = 0; j < R; ++j) {                          // fixed split order => deterministic
            const float *tj = cluster.map_shared_rank(tri, j);
            const float Mj = tj[hs];
            const float w = (Mj == -INFINITY) ? 0.0f : expf(Mj - MM);
            Lsum = fmaf(w, tj[hs + 1], Lsum);
            if (tid < hs) a2 = fmaf(w, tj[tid], a2);
        }
        if (tid < hs) xbs[tid] = a2 / Lsum;                    // softmax normalisation, :703-705
    }
    cluster.sync();                                            // peers are done reading this CTA's triple

    // ---- this CTA's rows of wo[:, h*hs:(h+1)*hs] . xb_h
    const float4 *xb4 = reinterpret_cast<const float4 *>(xbs);
    bool first = true;
    for (int rb = r0 + warp * RPW; rb < r1; rb += NG) {        // warp-uniform bound
        const int row = rb + rw;
        const bool valid = row < r1;
        float a = 0.0f;
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            const float4 w = first ? wpre[f]
                                   : (valid ? ldg_stream(wo4 + (size_t)row * q4 + lr + f * LPR) : make_float4(0.f, 0.f, 0.f, 0.f));
            a = dot4(w, xb4[lr + f * LPR], a);
        }
        first = false;
        for (int o = LPR >> 1; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (valid && lr == 0) q.parts[(size_t)h * q.dim + row] = a;
    }
}

// ---------------------------------------------------------------------------------------
// Small kernels
// ---------------------------------------------------------------------------------------
// End of one step of the on-device temperature-0 loop (src/main.zig:999-1041):
// choose next = forced[step] or argmax, record it, stop on BOS, advance (token, pos).
// Tensor parallel (world > 1): every rank first sends its local packed maximum to every rank as
// two LL units and takes the maximum of all of them, so all ranks advance with the same token
// without a collective launch.
struct AdvanceParams {
    int *ctl;
    unsigned long long *amax;
    const int *forced;
    int *out_next, *n_done;
    int world, rank;
    unsigned long long *ll_out[MAX_TP];   // rank d's landing area for my key: 2 units
    const unsigned long long *ll_in;      // my landing area: [world][2] units
    unsigned long long spin_ns;
};
__global__ void advance_kernel(const AdvanceParams p) {
    pdl_wait();
    int *ctl = p.ctl;
    if (ctl[CTL_DONE]) return;
    const int tid = threadIdx.x;
    __shared__ unsigned long long keys[MAX_TP];
    unsigned long long key = *p.amax;
    if (p.world > 1) {
        const unsigned int epoch = (unsigned int)ctl[CTL_EPOCH];
        if (tid < p.world)
            ll_store2(p.ll_out[tid], __uint_as_float((unsigned int)(key >> 32)),
                      __uint_as_float((unsigned int)(key & 0xFFFFFFFFull)), epoch);
        if (tid < p.world) {
            SpinGuard sg = spin_guard(ctl, p.spin_ns);
            uint4 a = ll_load2(p.ll_in + 2 * tid);
            while (a.y != epoch || a.w != epoch) {
                if (sg.expired()) break;
                a = ll_load2(p.ll_in + 2 * tid);
            }
            keys[tid] = ((unsigned long long)a.x << 32) | (unsigned long long)a.z;
        }
        __syncthreads();
        if (tid == 0)
            for (int r = 0; r < p.world; ++r) key = keys[r] > key ? keys[r] : key;
    }
    if (tid != 0) return;
    const int step = ctl[CTL_STEP];
    int next = (int)(0xFFFFFFFFu - (unsigned int)(key & 0xFFFFFFFFull));
    if (p.forced && p.forced[step] >= 0) next = p.forced[step];
    p.out_next[step] = next;
    *p.n_done = step + 1;
    *p.amax = 0ull;
    if (ctl[CTL_STOP_ON_BOS] && next == 1) {   // :1017-1019
        ctl[CTL_DONE] = 1;
        return;
    }
    ctl[CTL_TOKEN] = next;
    ctl[CTL_POS] = ctl[CTL_POS] + 1;
    ctl[CTL_STEP] = step + 1;
}

// advance_kernel for n decode streams stepping together (thread k = stream k): the forced token or
// the stream's own argmax (amax[k], packed by the classifier's EPI_ARGMAX epilogue), recorded at
// out_next[k * stride + step].  A stream that emits BOS with stop-on-BOS, or has taken its `limit`
// steps, is marked done; every later kernel of the loop skips it.
__global__ void advance_batch_kernel(BatchVec *vec, int n, unsigned long long *amax, const int *forced,
                                     int *out_next, int *n_done, int stride, int stop_on_bos) {
    pdl_wait();
    const int k = threadIdx.x;
    if (k >= n) return;
    BatchVec &v = vec[k];
    if (v.done) return;
    const unsigned long long key = amax[k];
    amax[k] = 0ull;
    const int step = v.step;
    int next = (int)(0xFFFFFFFFu - (unsigned int)(key & 0xFFFFFFFFull));
    if (forced && forced[k * stride + step] >= 0) next = forced[k * stride + step];
    out_next[k * stride + step] = next;
    n_done[k] = step + 1;
    if ((stop_on_bos && next == 1) || step + 1 >= v.limit) {   // :1017-1019
        v.done = 1;
        return;
    }
    v.token = next;
    v.pos = v.pos + 1;
    v.step = step + 1;
}

// Tensor parallel logits: every rank's classifier sent its vocab slice as LL units (EPI_XCHG with
// row_base = rank * vocab_loc); this kernel waits for all of them and writes the dense logits
// vector the D2H copy (and the sampler) read.  No collective launch per token.
__global__ void __launch_bounds__(NT) gather_logits_kernel(float *logits, const unsigned long long *ll_in,
                                                           int vocab, const int *ctl, unsigned long long spin_ns) {
    pdl_wait();
    if (ctl[CTL_DONE]) return;
    const unsigned int epoch = (unsigned int)ctl[CTL_EPOCH];
    SpinGuard sg = spin_guard(ctl, spin_ns);
    const int npairs = vocab >> 1;                          // vocab / world is even (checked at create)
    for (int i = blockIdx.x * NT + threadIdx.x; i < npairs; i += gridDim.x * NT) {
        uint4 a = ll_load2(ll_in + 2 * (size_t)i);
        while (a.y != epoch || a.w != epoch) {
            if (sg.expired()) break;
            a = ll_load2(ll_in + 2 * (size_t)i);
        }
        reinterpret_cast<float2 *>(logits)[i] = make_float2(__uint_as_float(a.x), __uint_as_float(a.z));
    }
}

// NCCL baseline mode (L2B_TP=nccl) only: x += all-reduced delta, the residual add of :395/:422
__global__ void __launch_bounds__(NT) resid_add_kernel(float *x, const float *delta, int n, const int *ctl) {
    if (ctl[CTL_DONE]) return;
    for (int i = blockIdx.x * NT + threadIdx.x; i < n; i += gridDim.x * NT) x[i] += delta[i];
}

// ---------------------------------------------------------------------------------------
// Sampler preparation on the device (src/main.zig:1005-1012, :752-768), SURVEY 8f.1: the part of
// temperature sampling that touches all vocab_size logits.  One CTA:
//   logits /= temperature (:1006); softmax in place (:1008, :687-706: max, exp, sum, divide);
//   top-p prefilter (:761-768): candidates with prob >= (1-p)/(n-1), compacted IN INDEX ORDER.
// The random draw, the sort of the (few) candidates and the CDF walk stay on the host because they
// use the host's PRNG (:730, :788).  temperature / top-p come from ctl[CTL_TEMP] / ctl[CTL_TOPP].
// ---------------------------------------------------------------------------------------
constexpr int SAMP_THREADS = 1024;
struct ProbIndex { float prob; int index; };
__global__ void __launch_bounds__(SAMP_THREADS) sample_prep_kernel(float *logits, int n, const int *ctl,
                                                                   ProbIndex *cand, int cand_cap, int *n_cand) {
    pdl_wait();
    if (ctl[CTL_DONE]) return;
    __shared__ float red[SAMP_THREADS / 32 + 1];
    __shared__ int wsum[SAMP_THREADS / 32 + 1];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float temp = __int_as_float(ctl[CTL_TEMP]);
    const float top_p = __int_as_float(ctl[CTL_TOPP]);
    // pass 1: scaled logits and their maximum
    float m = -INFINITY;
    for (int i = tid; i < n; i += SAMP_THREADS) {
        const float v = __fdiv_rn(logits[i], temp);         // :1006
        logits[i] = v;
        m = fmaxf(m, v);
    }
    m = warp_max(m);
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = red[lane];                                           // 32 warps
    m = warp_max(m);
    __syncthreads();
    // pass 2: exp and sum
    float l = 0.0f;
    for (int i = tid; i < n; i += SAMP_THREADS) {
        const float e = expf(logits[i] - m);                 // :699
        logits[i] = e;
        l += e;
    }
    l = warp_sum(l);
    if (lane == 0) red[warp] = l;
    __syncthreads();
    l = red[lane];
    l = warp_sum(l);
    __syncthreads();
    // pass 3: normalise (:703-705) and select candidates; thread t owns a CONTIGUOUS index range so
    // that an exclusive scan of the per-thread counts yields index-ordered compaction
    const int per = (n + SAMP_THREADS - 1) / SAMP_THREADS;
    const int i0 = tid * per, i1 = min(n, i0 + per);
    const float cutoff = __fdiv_rn(1.0f - top_p, (float)n - 1.0f);   // :761
    int cnt = 0;
    for (int i = i0; i < i1; ++i) {
        const float pr = __fdiv_rn(logits[i], l);
        logits[i] = pr;
        if (top_p >= 0.0f && pr >= cutoff) ++cnt;            // :764
    }
    if (top_p < 0.0f) { if (tid == 0) *n_cand = -1; return; }
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = wsum[lane];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        wsum[lane] = wi - w;                                 // exclusive prefix of the warp totals
        if (lane == 31) *n_cand = wi;
    }
    __syncthreads();
    int off = wsum[warp] + incl - cnt;
    for (int i = i0; i < i1; ++i) {
        const float pr = logits[i];
        if (pr >= cutoff) {
            if (off < cand_cap) { cand[off].prob = pr; cand[off].index = i; }
            ++off;
        }
    }
}

// standalone rmsnorm (unit-test surface; the hot path fuses it into the GEMV prologue)
__global__ void __launch_bounds__(NT) rmsnorm_kernel(float *o, const float *x, const float *w, int n) {
    __shared__ float scratch[NWARP + 1];
    float ssq = 0.0f;
    for (int i = threadIdx.x; i < n; i += NT) ssq = fmaf(x[i], x[i], ssq);
    float ss = block_sum(ssq, scratch);
    ss /= (float)n;
    ss += 1e-5f;
    const float s = 1.0f / sqrtf(ss);
    for (int i = threadIdx.x; i < n; i += NT) o[i] = __fmul_rn(__fmul_rn(x[i], s), w[i]);
}

// standalone softmax (:687-706) over n values in global memory, one CTA (unit-test surface)
__global__ void __launch_bounds__(NT) softmax_kernel(float *x, int n) {
    __shared__ float scratch[NWARP + 1];
    float m = -INFINITY;
    for (int i = threadIdx.x; i < n; i += NT) m = fmaxf(m, x[i]);
    m = block_max(m, scratch);
    float l = 0.0f;
    for (int i = threadIdx.x; i < n; i += NT) {
        const float e = expf(x[i] - m);
        x[i] = e;
        l += e;
    }
    l = block_sum(l, scratch);
    for (int i = threadIdx.x; i < n; i += NT) x[i] = x[i] / l;
}

// standalone vector_weighted_sum_rows (:657-685), arbitrary out_len / stride (unit-test surface)
__global__ void __launch_bounds__(NT) weighted_rows_kernel(float *xout, int out_len, const float *rows,
                                                           int row_stride, const float *weights,
                                                           int n_weights) {
    for (int i = blockIdx.x * NT + threadIdx.x; i < out_len; i += gridDim.x * NT) {
        float s = 0.0f;
        for (int r = 0; r < n_weights; ++r) s = fmaf(rows[(size_t)r * row_stride + i], weights[r], s);
        xout[i] = s;
    }
}

// ---------------------------------------------------------------------------------------
// Synthetic weights: counter-based, integer-only hash so CPU and GPU agree bit for bit.
// ---------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return z;
}
__host__ __device__ __forceinline__ int32_t synth_irwin_hall(uint64_t tensor_seed, uint64_t i) {
    const uint64_t h = mix64(tensor_seed + (i + 1) * 0x9E3779B97F4A7C15ull);
    return (int32_t)((h & 0xFFFF) + ((h >> 16) & 0xFFFF) + ((h >> 32) & 0xFFFF) + ((h >> 48) & 0xFFFF)) -
           131070;
}
// rows x cols window of a (.., src_cols) tensor starting at element `first`, written densely
__global__ void synth_fill_kernel(float *dst, uint64_t rows, uint64_t cols, uint64_t first,
                                  uint64_t src_cols, uint64_t tensor_seed, double mean, double scale,
                                  float lo, float hi) {
    const uint64_t total = rows * cols;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < total;
         j += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = j / cols, c = j - r * cols;
        const uint64_t i = first + r * src_cols + c;
        const int32_t s = synth_irwin_hall(tensor_seed, i);
        float v = (float)__dadd_rn(__dmul_rn((double)s, scale), mean);
        v = fminf(fmaxf(v, lo), hi);
        dst[j] = v;
    }
}

}  // namespace l2b
