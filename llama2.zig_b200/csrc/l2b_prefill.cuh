// l2b_prefill.cuh — batched passes over the weights: NB activation vectors share one pass.  They are
// consecutive positions of one prompt (prefill, SURVEY 8f.2) or one token of each of NB decode
// streams over the same weights (l2b_forward_batch / l2b_generate_argmax_batch); each vector takes
// its token, position and KV cache from a BatchVec table in device memory.
//
// The reference feeds prompt tokens through transformer() one at a time (src/main.zig:996-1000) and
// streams every weight once per token.  For bandwidth-bound shapes (llama2-7B) the same streaming
// kernel as the decode step (gemv_tma_kernel: TMA ring, warp-specialised producer / consumers /
// epilogue) carries NB activation vectors instead of one: each 128-bit weight load feeds NB x 4
// FMAs, so the weight traffic per prompt token drops NB-fold while fp32 CUDA-core arithmetic stays
// far below its roof (NB = 4: 2 flop/B).  Per (row, position) the summation order is the decode
// kernel's own — same thread-to-column mapping, same butterfly, same fixed-order combine — so a
// prefilled position holds what the token-by-token path would have computed.
#pragma once

#include "l2b_device.cuh"

namespace l2b {

constexpr int PF_MAXB = 4;

struct PrefillParams {
    // ---- input vectors: NB contiguous vectors of n floats, or (layer 0) embedding rows of vec[b].token
    const float *x_in;
    const float *emb;
    const BatchVec *vec;    // device table: the pass's vectors (token, position, KV cache, done)
    const float *gamma;     // rmsnorm gain => fused rmsnorm of every vector
    float *x_out;           // layer 0: CTA 0 writes the NB embedding rows here (the residual-stream batch)
    int n, nb;              // columns; positions in this chunk (<= NB)
    // ---- matrices
    const float *w0, *w1, *w2;
    int rows0, rows1, rows2, total_rows;
    // ---- outputs: EPI_QKV: q batch [nb][rows0]; EPI_SILU: hb batch [nb][rows0]; EPI_RESID: x batch
    // [nb][total_rows]; EPI_STORE / EPI_ARGMAX: logits batch [nb][total_rows]
    float *out0;
    unsigned long long *amax;           // EPI_ARGMAX: packed argmax key of vector b at amax[b]
    size_t kv_off;                      // EPI_QKV: this layer's offset in vec[b].kc / vc ((seq_len, kv_dim) per layer)
    const float *rope_cos, *rope_sin;   // (seq_len, head_size/2)
    int head_size, kv_dim;
    int nstage;
};

// transposing butterfly of the decode kernel: 8 per-row partials across the 32 lanes; afterwards
// lane L (L % 4 == 0) holds the warp's sum of row L / 4 in a[0]
__device__ __forceinline__ void butterfly8(float (&a)[GEMV8_R], int lane) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float send = (lane & 16) ? a[i] : a[i + 4];
        const float keep = (lane & 16) ? a[i + 4] : a[i];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float send = (lane & 8) ? a[i] : a[i + 2];
        const float keep = (lane & 8) ? a[i + 2] : a[i];
        a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
    {
        const float send = (lane & 4) ? a[0] : a[1];
        const float keep = (lane & 4) ? a[1] : a[0];
        a[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    a[0] += __shfl_xor_sync(0xffffffffu, a[0], 2);
    a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
}

template <int EPI>
__device__ __forceinline__ const float *pf_row_ptr(const PrefillParams &p, int v) {
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

template <int EPI, int NB>
__global__ void __launch_bounds__(TMA_THREADS, 1) prefill_gemm_kernel(const PrefillParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int NSTAGE = p.nstage;
    float *ring = reinterpret_cast<float *>(smem_raw);                 // NSTAGE x 32 KB
    float *xs = ring + (size_t)NSTAGE * TMA_STAGE_FLOATS;              // NB x n floats
    __shared__ uint64_t full[TMA_MAX_STAGES], empty[TMA_MAX_STAGES], xbar, tile_full[2], tile_free[2];
    __shared__ float scratch[NB][NWARP + 2];
    __shared__ float red[2][NWARP][GEMV8_R][NB];
    __shared__ float rope_s[NB][2][128];                               // cos/sin rows of the vectors' positions

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n4 = p.n >> 2;
    const int nsteps = (n4 + NT - 1) / NT;
    const int npairs = (p.total_rows + 1) >> 1;
    const int base = npairs / (int)gridDim.x, rem = npairs % (int)gridDim.x;
    const int b0 = blockIdx.x;
    const int pair0 = b0 * base + min(b0, rem);
    const int pair1 = pair0 + base + (b0 < rem ? 1 : 0);
    const int r0 = pair0 * 2, r1 = min(pair1 * 2, p.total_rows);
    const int ntiles = (r1 - r0 + GEMV8_R - 1) / GEMV8_R;
    const int total = ntiles * nsteps;

    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], NWARP); }
        mbar_init(&xbar, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&tile_full[s], NWARP); mbar_init(&tile_free[s], 1); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == NWARP) {
        // ---- producer warp (identical to the decode kernel's): lane r issues row r's bulk copy
        int p_it = 0, p_stage = 0, p_tile = 0, p_step = 0;
        uint32_t p_phase = 0;
        const float *p_row = nullptr;
        while (p_it < total) {
            const int c0 = p_step * NT;
            const int cols4 = min(NT, n4 - c0);
            const int v0 = r0 + p_tile * GEMV8_R;
            const int rows = min(GEMV8_R, r1 - v0);
            if (p_step == 0 && lane < rows) p_row = pf_row_ptr<EPI>(p, v0 + lane);
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
        }
        pdl_launch_dependents();
        return;
    }

    // ---- prologue (consumer warps + epilogue warp; named barrier 1)
    constexpr int MAXV = 5;
    constexpr int PRO_THREADS = TMA_THREADS - 32;
    const int ptid = tid < NT ? tid : tid - 32;
    float4 gv[MAXV];
    if (p.gamma) {
        const float4 *g4 = reinterpret_cast<const float4 *>(p.gamma);
#pragma unroll
        for (int k = 0; k < MAXV; ++k) {
            const int i = ptid + k * PRO_THREADS;
            gv[k] = (i < n4) ? __ldg(g4 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    pdl_wait();
    {
        if (tid == 0) {
            const uint32_t bytes = (uint32_t)p.n * 4u;
            mbar_expect_tx(&xbar, bytes * (uint32_t)p.nb);
            if (p.emb) {
                for (int b = 0; b < p.nb; ++b)                          // x[b] = token_embedding_table[token], :295-296
                    tma_load_1d(xs + (size_t)b * p.n, p.emb + (size_t)p.vec[b].token * p.n, bytes, &xbar);
            } else {
                tma_load_1d(xs, p.x_in, bytes * (uint32_t)p.nb, &xbar);
            }
        }
        if (EPI == EPI_QKV && tid >= NT + 32) {                        // epilogue warp: RoPE rows of the vectors' positions
            const int half = p.head_size >> 1;
            for (int b = 0; b < p.nb; ++b) {
                const int pos = p.vec[b].pos;
                for (int i = lane; i < half; i += 32) {
                    rope_s[b][0][i] = __ldg(p.rope_cos + (size_t)pos * half + i);
                    rope_s[b][1][i] = __ldg(p.rope_sin + (size_t)pos * half + i);
                }
            }
        }
        mbar_wait(&xbar, 0);
        if (p.gamma || p.x_out) {
            float4 *xs4w = reinterpret_cast<float4 *>(xs);
            float ssq[NB];
#pragma unroll
            for (int b = 0; b < NB; ++b) {
                ssq[b] = 0.0f;
                if (b < p.nb) {
#pragma unroll
                    for (int k = 0; k < MAXV; ++k) {
                        const int i = ptid + k * PRO_THREADS;
                        if (i < n4) {
                            const float4 v = xs4w[(size_t)b * n4 + i];
                            if (p.x_out && blockIdx.x == 0) reinterpret_cast<float4 *>(p.x_out)[(size_t)b * n4 + i] = v;
                            ssq[b] = fmaf(v.x, v.x, ssq[b]); ssq[b] = fmaf(v.y, v.y, ssq[b]);
                            ssq[b] = fmaf(v.z, v.z, ssq[b]); ssq[b] = fmaf(v.w, v.w, ssq[b]);
                        }
                    }
                }
            }
            if (p.gamma) {
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    const float w = warp_sum(ssq[b]);
                    if (lane == 0) scratch[b][ptid >> 5] = w;
                }
                named_bar_sync(1, PRO_THREADS);
#pragma unroll
                for (int b = 0; b < NB; ++b) {
                    if (b >= p.nb) continue;
                    float ss = (lane < PRO_THREADS / 32) ? scratch[b][lane] : 0.0f;
                    ss = warp_sum(ss);
                    ss /= (float)p.n;            // :452
                    ss += 1e-5f;                 // :453
                    const float sc = 1.0f / sqrtf(ss);  // :454
#pragma unroll
                    for (int k = 0; k < MAXV; ++k) {
                        const int i = ptid + k * PRO_THREADS;
                        if (i < n4) {
                            float4 v = xs4w[(size_t)b * n4 + i];
                            v.x = __fmul_rn(__fmul_rn(v.x, sc), gv[k].x);   // (x*s)*w, :462
                            v.y = __fmul_rn(__fmul_rn(v.y, sc), gv[k].y);
                            v.z = __fmul_rn(__fmul_rn(v.z, sc), gv[k].z);
                            v.w = __fmul_rn(__fmul_rn(v.w, sc), gv[k].w);
                            xs4w[(size_t)b * n4 + i] = v;
                        }
                    }
                }
            }
        }
        named_bar_sync(1, PRO_THREADS);
    }

    if (warp == NWARP + 1) {
        // ---- epilogue warp: lane = b * 4 + pair handles (row pair, position b) of each tile
        // (a vector whose generation has ended writes nothing: no KV append, no residual update)
        const int eb = lane >> 2, ep = lane & 3;
        const bool active = lane < 4 * NB && eb < p.nb && !p.vec[eb].done;
        int pos = 0;
        float *kc = nullptr, *vc = nullptr;
        if (EPI == EPI_QKV && active) { pos = p.vec[eb].pos; kc = p.vec[eb].kc + p.kv_off; vc = p.vec[eb].vc + p.kv_off; }
        unsigned long long best = 0ull;
        for (int t = 0; t < ntiles; ++t) {
            const int par = t & 1, use = t >> 1;
            mbar_wait(&tile_full[par], use & 1);
            float s0 = 0.0f, s1 = 0.0f;
            if (lane < 4 * NB) {
#pragma unroll
                for (int w8 = 0; w8 < NWARP; ++w8) {       // fixed order
                    s0 += red[par][w8][2 * ep][eb];
                    s1 += red[par][w8][2 * ep + 1][eb];
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&tile_free[par]);
            const int vp = r0 + t * GEMV8_R + 2 * ep;
            if (!active || vp >= r1) continue;
            if (EPI == EPI_QKV) {
                if (vp < p.rows0 + p.rows1) {
                    const bool is_q = vp < p.rows0;
                    const int i = is_q ? vp : vp - p.rows0;
                    const int pr = (i % p.head_size) >> 1;                                  // :338
                    const float fcr = rope_s[eb][0][pr], fci = rope_s[eb][1][pr];
                    const float q0 = __fsub_rn(__fmul_rn(s0, fcr), __fmul_rn(s1, fci));      // :348
                    const float q1 = __fadd_rn(__fmul_rn(s0, fci), __fmul_rn(s1, fcr));      // :349
                    float *dst = is_q ? p.out0 + (size_t)eb * p.rows0 + i : kc + (size_t)pos * p.kv_dim + i;   // :355,:357
                    *reinterpret_cast<float2 *>(dst) = make_float2(q0, q1);
                } else {
                    const int i = vp - p.rows0 - p.rows1;
                    *reinterpret_cast<float2 *>(vc + (size_t)pos * p.kv_dim + i) = make_float2(s0, s1);   // :356,:358
                }
            } else if (EPI == EPI_SILU) {
                const float sg = __fmul_rn(s0, __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-s0))));   // :412
                p.out0[(size_t)eb * p.rows0 + (vp >> 1)] = __fmul_rn(sg, s1);                  // :416
            } else if (EPI == EPI_STORE || EPI == EPI_ARGMAX) {   // logits row b (:429)
                float *dst = p.out0 + (size_t)eb * p.total_rows + vp;
                dst[0] = s0;
                if (vp + 1 < p.total_rows) dst[1] = s1;
                if (EPI == EPI_ARGMAX) {   // first maximum wins (:715-726), as gemv_epilogue_pair
                    const unsigned long long k0 = argmax_key(s0, vp);
                    best = k0 > best ? k0 : best;
                    if (vp + 1 < p.total_rows) {
                        const unsigned long long k1 = argmax_key(s1, vp + 1);
                        best = k1 > best ? k1 : best;
                    }
                }
            } else {   // EPI_RESID: x[b][row] += acc (:395, :422)
                float *dst = p.out0 + (size_t)eb * p.total_rows + vp;
                if (vp + 1 < p.total_rows) {
                    const float2 o = *reinterpret_cast<const float2 *>(dst);
                    *reinterpret_cast<float2 *>(dst) = make_float2(o.x + s0, o.y + s1);
                } else {
                    dst[0] += s0;
                }
            }
        }
        if (EPI == EPI_ARGMAX) {   // the 4 lanes of vector b, then one 64-bit atomicMax per CTA and vector
            best = max(best, __shfl_xor_sync(0xffffffffu, best, 1));
            best = max(best, __shfl_xor_sync(0xffffffffu, best, 2));
            if (active && ep == 0 && best) atomicMax(p.amax + eb, best);
        }
        return;
    }

    // ---- consumers (warps 0..7): NB accumulator sets per row
    const float4 *xs4 = reinterpret_cast<const float4 *>(xs);
    float acc[NB][GEMV8_R];
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
        for (int r = 0; r < GEMV8_R; ++r) acc[b][r] = 0.0f;
    int c_stage = 0;
    uint32_t c_phase = 0;
    int t = 0, st = 0;
    for (int it = 0; it < total; ++it, ++st) {
        if (st == nsteps) { st = 0; ++t; }
        const int c = st * NT + tid;
        const int v0 = r0 + t * GEMV8_R;
        const int rows = min(GEMV8_R, r1 - v0);
        mbar_wait(&full[c_stage], c_phase);
        if (c < n4) {
            const float4 *w4 = reinterpret_cast<const float4 *>(ring + (size_t)c_stage * TMA_STAGE_FLOATS) + tid;
            float4 xv[NB];
#pragma unroll
            for (int b = 0; b < NB; ++b) xv[b] = xs4[(size_t)(b < p.nb ? b : 0) * n4 + c];
#pragma unroll
            for (int r = 0; r < GEMV8_R; ++r) {
                if (r < rows) {
                    const float4 w = w4[r * NT];
#pragma unroll
                    for (int b = 0; b < NB; ++b) acc[b][r] = dot4(w, xv[b], acc[b][r]);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[c_stage]);
        if (++c_stage == NSTAGE) { c_stage = 0; c_phase ^= 1; }
        if (st != nsteps - 1) continue;
#pragma unroll
        for (int b = 0; b < NB; ++b) butterfly8(acc[b], lane);
        const int par = t & 1, use = t >> 1;
        mbar_wait(&tile_free[par], (use & 1) ^ 1);
        if ((lane & 3) == 0) {
#pragma unroll
            for (int b = 0; b < NB; ++b) red[par][warp][lane >> 2][b] = acc[b][0];
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&tile_full[par]);
#pragma unroll
        for (int b = 0; b < NB; ++b)
#pragma unroll
            for (int r = 0; r < GEMV8_R; ++r) acc[b][r] = 0.0f;
    }
}

}  // namespace l2b
