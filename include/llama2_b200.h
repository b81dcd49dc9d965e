/*
 * llama2_b200.h — C ABI of the B200 (sm_100a) decode hot path for cgbur/llama2.zig.
 *
 * This library replaces ONE internal call of the reference,
 *     transformer(token, pos, &config, &state, &weights)      src/main.zig:285, call site :996
 * and the numeric helpers it calls (src/main.zig:432-713).  The reference has no FFI of
 * its own; these entry points are what its Zig host declares `extern "c"` (see
 * INTEGRATION.md for the patch).  Everything else (CLI, checkpoint and tokenizer
 * loaders, sampler) stays in the host.
 *
 * Conventions
 *   - plain C types only; every call returns L2B_OK (0) or a negative l2b_status and never
 *     aborts or throws across the boundary (the reference's `assert`s, e.g. :433-434,
 *     :534-540, become argument checks);
 *   - host pointers are borrowed for the duration of the call only;
 *   - one context = one decode stream on 1, 2, 4 or 8 GPUs; not thread-safe (the reference is
 *     single-threaded); contexts that share one set of weights (l2b_create_stream) are driven
 *     from one thread, like a single context;
 *   - there is NO CPU fallback: if no sm_100 device is usable the call fails with
 *     L2B_ERR_CUDA / L2B_ERR_NO_DEVICE.
 */
#ifndef LLAMA2_B200_H
#define LLAMA2_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define L2B_ABI_VERSION 2

typedef enum l2b_status {
    L2B_OK = 0,
    L2B_ERR_INVALID_ARG = -1,   /* NULL pointer, token/pos out of range, bad size          */
    L2B_ERR_UNSUPPORTED = -2,   /* shape the kernels do not cover (see l2b_create)          */
    L2B_ERR_CUDA = -3,          /* a CUDA runtime call failed; see l2b_last_error()         */
    L2B_ERR_NO_DEVICE = -4,     /* no CUDA device / not compute capability 10.x             */
    L2B_ERR_OOM = -5,           /* device or pinned-host allocation failed                  */
    L2B_ERR_COMM = -6,          /* peer-memory setup failed, or a tensor-parallel peer timed out */
    L2B_ERR_STATE = -7          /* call order violated (e.g. pos beyond what was appended)  */
} l2b_status;

/* Mirrors ConfigReader (src/main.zig:17-25) after main() has normalised it (:942-946):
 * vocab_size is already abs(), shared_weights = (header vocab_size > 0).                 */
typedef struct l2b_config {
    int32_t dim;            /* transformer dimension                                       */
    int32_t hidden_dim;     /* ffn hidden dimension                                        */
    int32_t n_layers;
    int32_t n_heads;
    int32_t n_kv_heads;     /* < n_heads for multi-query / grouped-query (:291, :314-320)  */
    int32_t vocab_size;
    int32_t seq_len;
    int32_t shared_weights; /* 1: classifier == token embedding table (:112)               */
} l2b_config;

/* Tensor-parallel placement of one context (BASELINE.json config 5; SURVEY.md 8e).
 * world_size == 1 means the whole model on `device`.  For world_size in {2,4,8}
 * wq/wk/wv/w1/w3/wcls are split by output rows, wo/w2 by input columns, and the hidden
 * vector is all-reduced after wo and after w2 (inside the GEMV kernels, over NVLink peer
 * memory).  Two ways to get there:
 *   - ONE process, l2b_create(..., n_gpus): what the Zig CLI uses (`--gpus N`); nothing else
 *     changes for the caller, every l2b_* call drives all GPUs;
 *   - one process PER GPU, l2b_create_sharded with this struct: the caller moves `comm_id` (from
 *     l2b_comm_unique_id on rank 0) to every rank by its own means (bench.py uses
 *     torch.distributed) and every rank makes the same calls in the same order (lockstep: each
 *     decode step exchanges data with every other rank; a rank that stops stepping makes the
 *     others return L2B_ERR_COMM after a bounded wait, L2B_SPIN_TIMEOUT_MS, default 20 s).      */
typedef struct l2b_shard {
    int32_t rank;
    int32_t world_size;
    int32_t device;          /* CUDA device ordinal for this context                        */
    int32_t reserved;
    uint8_t comm_id[128];    /* opaque rendezvous token; ignored when world_size == 1       */
} l2b_shard;

typedef struct l2b_ctx l2b_ctx;

/* ---- lifecycle ---------------------------------------------------------------------- */

/* Replaces Weights.init (src/main.zig:73-115) + RunState.init (:137-154) on the device.
 *   host_weights : the checkpoint payload after the 28-byte header, exactly the `data`
 *                  buffer of src/main.zig:955-967, laid out as :85-112; n_floats its length.
 *   rope_cos/sin : optional (seq_len, head_size/2) tables the host computed with the
 *                  expressions of :338-342 (so RoPE is bit-identical to the host's libm);
 *                  NULL => the library computes them with the same expressions.
 *   n_gpus       : 1, 2, 4 or 8 GPUs (devices 0..n_gpus-1) driven by this one process; for
 *                  n_gpus > 1 the model is sharded as described at l2b_shard and the GPUs must
 *                  be NVLink peers.  The upload streams through pinned double buffers
 *                  (see l2b_load_stats).
 * Supported shapes: dim % 4 == 0, hidden_dim % 4 == 0, head_size = dim/n_heads a multiple of
 * 4 and <= 256, n_heads % n_kv_heads == 0; for n_gpus > 1 also n_kv_heads, hidden_dim/4 and
 * vocab_size/2 divisible by n_gpus.  Anything else => L2B_ERR_UNSUPPORTED.                  */
int32_t l2b_create(l2b_ctx **out, const l2b_config *cfg, const float *host_weights,
                   uint64_t n_floats, const float *rope_cos, const float *rope_sin,
                   int32_t n_gpus);

/* Same, for one tensor-parallel rank.  host_weights is the FULL payload; the library
 * uploads only this rank's slices.                                                         */
int32_t l2b_create_sharded(l2b_ctx **out, const l2b_config *cfg, const float *host_weights,
                           uint64_t n_floats, const float *rope_cos, const float *rope_sin,
                           const l2b_shard *shard);

/* Synthetic checkpoint of the given shape generated directly in device memory
 * (SURVEY.md 8d: stories110M / llama2-7B are not shipped; a 27 GB file is impractical).
 * The generator is a counter-based integer hash, bit-identical to
 * l2b_synth_fill_host() below, so a CPU checker can materialise the same weights.
 * shard may be NULL (single GPU, device 0).                                                */
int32_t l2b_create_synthetic(l2b_ctx **out, const l2b_config *cfg, uint64_t seed,
                             const l2b_shard *shard);
/* Same weights, one process driving n_gpus GPUs (the synthetic twin of l2b_create(.., n_gpus)). */
int32_t l2b_create_synthetic_group(l2b_ctx **out, const l2b_config *cfg, uint64_t seed,
                                   int32_t n_gpus);

void l2b_destroy(l2b_ctx *ctx);

/* Forget the KV cache (start a new generation at pos 0).  The reference runs one
 * generation per process and has no such entry point; benches need it.                     */
int32_t l2b_reset(l2b_ctx *ctx);

/* ---- the hot path ------------------------------------------------------------------- */

/* transformer(token, pos, ...) of src/main.zig:285-430.  On return host_logits[0..vocab)
 * holds what the reference leaves in state.logits (:429); the caller may then mutate it
 * exactly as :1002-1013 do.  pos must be 0 on the first call and may not skip ahead:
 * pos <= (number of positions appended so far).  Synchronous.                               */
int32_t l2b_forward(l2b_ctx *ctx, int32_t token, int32_t pos, float *host_logits);

/* Same step, but the argmax of :715-726 (first maximum wins) runs on the device in the
 * classifier epilogue and only the token id crosses PCIe.  The `-t 0` path (:1002-1003).   */
int32_t l2b_forward_argmax(l2b_ctx *ctx, int32_t token, int32_t pos, int32_t *next);

/* Zero-copy variant: runs the step and returns a pointer to the library's pinned host
 * buffer of vocab_size logits (valid until the next call on this context).                 */
int32_t l2b_forward_pinned(l2b_ctx *ctx, int32_t token, int32_t pos, const float **logits);

/* The library's pinned logits buffer (vocab_size floats, lives as long as the context).  A host
 * that uses it AS state.logits (src/main.zig:149: `state.logits = l2b_logits_buffer(ctx)[0..V]`)
 * and passes it to l2b_forward gets the logits with no second host copy: the D2H DMA of the step
 * lands directly in it.                                                                    */
float *l2b_logits_buffer(l2b_ctx *ctx);

/* transformer() + the vocab-wide part of temperature sampling (src/main.zig:1005-1012) on the
 * device: logits /= temperature (:1006), softmax (:1008), and for 0 < top_p < 1 the candidate
 * prefilter of sample_top_p (:761-768: prob >= (1-top_p)/(n-1), in index order).  The random
 * draw, the sort of the few candidates and the CDF walk stay on the host (they use the host's
 * PRNG, :730, :788).
 *   host_probs : vocab_size probabilities (what :1008 leaves in state.logits); may be NULL when
 *                only the candidates are wanted, or l2b_logits_buffer(ctx) for zero copy.
 *   cand/n_cand: for 0 < top_p < 1: *n_cand candidates (prob, index); if more than cand_cap (or
 *                8192) passed the filter, *n_cand = -(their number) and the host filters
 *                host_probs itself.  Ignored (may be NULL) for top_p == 0 or 1 (:1009).         */
typedef struct l2b_prob_index { float prob; int32_t index; } l2b_prob_index;
int32_t l2b_forward_sample(l2b_ctx *ctx, int32_t token, int32_t pos, float temperature, float top_p,
                           float *host_probs, l2b_prob_index *cand, int32_t cand_cap,
                           int32_t *n_cand);

/* Whole temperature-0 generation loop of src/main.zig:995-1042 on the device: starts from
 * `token` at position `pos`, runs up to n_steps steps, feeds forced[i] (if forced != NULL
 * and forced[i] >= 0, like prompt forcing :999-1000) or the on-device argmax back in, and
 * stops after emitting BOS (token 1, :1017-1019) when stop_on_bos != 0.  out_next[i] is the
 * token chosen at step i; *n_done the number of transformer steps executed.                */
int32_t l2b_generate_argmax(l2b_ctx *ctx, int32_t token, int32_t pos, int32_t n_steps,
                            const int32_t *forced, int32_t stop_on_bos, int32_t *out_next,
                            int32_t *n_done);

/* Prompt prefill (SURVEY.md 8f.2).  The reference feeds prompt tokens through transformer() one at
 * a time and discards their logits (src/main.zig:996-1000).  This runs positions pos0 ..
 * pos0+n_tokens-1 with tokens[i] at position pos0+i back to back on the device: no host round trip
 * per position, and the classifier is skipped for every position whose logits nobody reads.
 * host_logits == NULL: no logits at all (the KV cache is all the caller wants); otherwise the
 * logits of the LAST position are returned, exactly as l2b_forward would.  Per position the
 * arithmetic is the decode step's own, so KV cache and logits equal n_tokens calls of
 * l2b_forward bit for bit.                                                                 */
int32_t l2b_prefill(l2b_ctx *ctx, const int32_t *tokens, int32_t n_tokens, int32_t pos0,
                    float *host_logits);

/* ---- several decode streams over one copy of the weights ----------------------------- */

#define L2B_MAX_BATCH 8

/* A new decode stream over base's device weights: its own KV cache, run state, control block,
 * pinned buffers and graphs; no weight upload (l2b_load_stats reports 0 bytes).  Weights are
 * reference-counted: base may be destroyed before its streams.  Single-GPU contexts only (a
 * sharded or in-process-group base => L2B_ERR_UNSUPPORTED).  A stream is an ordinary l2b_ctx:
 * every existing call (forward, prefill, forward_sample, generate_argmax, reset, read_state...)
 * works on it unchanged.                                                                   */
int32_t l2b_create_stream(l2b_ctx **out, l2b_ctx *base);

/* One transformer() step for each of n streams (distinct, over the same weights,
 * 1 <= n <= L2B_MAX_BATCH): tokens[k] at pos[k] on streams[k]; host_logits is [n][vocab].  Per
 * stream the result equals l2b_forward on that stream alone.  On bandwidth-bound shapes (today
 * llama2-7B on one GPU) up to 4 streams share each pass over the weights; on every other shape the
 * streams' own steps run in turn (same results, no speed-up).
 * Errors: NULL pointers, n outside 1..L2B_MAX_BATCH, a stream listed twice, streams over different
 * weights, token or pos out of range => L2B_ERR_INVALID_ARG; pos[k] beyond what streams[k] has
 * appended => L2B_ERR_STATE.  l2b_last_timing(streams[0]) reports the device time and kernel
 * launches of the call; every stream's appended length is updated, so single-stream calls continue
 * any stream.  What l2b_read_state returns for x / xb / hb / q / logits of a stream after a batch
 * call is unspecified (its KV cache rows are exact).                                        */
int32_t l2b_forward_batch(l2b_ctx *const *streams, int32_t n, const int32_t *tokens,
                          const int32_t *pos, float *host_logits);

/* l2b_generate_argmax for n streams stepping together on the device, with no host round trip per
 * step.  forced is [n][n_steps] (or NULL; -1 = free-running), out_next is [n][n_steps], n_done is
 * [n].  Steps of stream k are clamped to seq_len - pos[k]; a stream that emits BOS with stop_on_bos
 * stops (its KV cache and outputs stay as the single-stream loop would leave them) while the others
 * continue.  Argument checks, timing and state as l2b_forward_batch.                        */
int32_t l2b_generate_argmax_batch(l2b_ctx *const *streams, int32_t n, const int32_t *tokens,
                                  const int32_t *pos, int32_t n_steps, const int32_t *forced,
                                  int32_t stop_on_bos, int32_t *out_next, int32_t *n_done);

/* ---- introspection ------------------------------------------------------------------- */

const char *l2b_last_error(const l2b_ctx *ctx);     /* never NULL                           */
const char *l2b_status_string(int32_t status);
int32_t l2b_abi_version(void);

/* Copies one RunState buffer (src/main.zig:119-135) of the last step to the host, for
 * layer-level parity tests: 0=x 1=xb 2=hb 3=q 4=key_cache 5=value_cache 6=logits.
 * Sharded contexts return this rank's slice.  n = capacity of dst in floats; *n_out the
 * floats written.                                                                          */
int32_t l2b_read_state(l2b_ctx *ctx, int32_t which, float *dst, uint64_t n, uint64_t *n_out);

/* Device time (ms, CUDA events on the context's stream) of the last l2b_generate_argmax /
 * l2b_prefill call (single steps are only timed when L2B_TIME_STEPS=1 is in the environment
 * at create time: the two event records cost the end-to-end loop of a small model ~3 %), and how
 * many kernels of this library the last call launched.                                      */
int32_t l2b_last_timing(const l2b_ctx *ctx, float *device_ms, int32_t *kernel_launches);

/* Checkpoint ingest of the last l2b_create on this context (SURVEY.md 8f.3): wall time of the
 * pinned, double-buffered upload of all weight tensors and the bytes it moved (rank 0's shard
 * for multi-GPU contexts).                                                                  */
int32_t l2b_load_stats(const l2b_ctx *ctx, double *upload_ms, uint64_t *upload_bytes);

/* Per-kernel device times of ONE step (eager launches with a CUDA event between kernels, on
 * the context's stream), for roofline accounting: `bytes` is the algorithmic traffic of that
 * launch (weight rows x columns x 4, or the K and V rows attention reads).  The step is a
 * real step (KV cache is appended, logits are produced).  out has room for cap entries;
 * *n_out receives the number of kernels in a step.                                          */
typedef struct l2b_kernel_time {
    char name[24];          /* "qkv_rope", "attention", "wo", "w13_silu", "w2", "classifier" */
    int32_t layer;          /* -1 for the classifier                                         */
    float ms;
    uint64_t bytes;
} l2b_kernel_time;
int32_t l2b_profile_step(l2b_ctx *ctx, int32_t token, int32_t pos, l2b_kernel_time *out,
                         int32_t cap, int32_t *n_out);

/* Debug: with L2B_TRACE=1 in the environment at l2b_create time, every kernel of a step stamps
 * %globaltimer at fixed points (entry, ring filled, dependency wait done, activations staged,
 * first/last stage consumed, producer done, epilogue done).  Copies the last step's table
 * [launch][512 CTAs][8 slots] (ns) to dst.                                                  */
int32_t l2b_debug_trace(l2b_ctx *ctx, unsigned long long *dst, uint64_t cap_words, uint64_t *n_words);

/* Algorithmic bytes one step at position pos must read (SURVEY.md 8d):
 * weight bytes (this rank's shard) and KV-cache bytes.                                     */
int32_t l2b_step_bytes(const l2b_ctx *ctx, int32_t pos, uint64_t *weight_bytes,
                       uint64_t *kv_bytes);

/* ---- multi-GPU rendezvous -------------------------------------------------------------- */
int32_t l2b_comm_unique_id(uint8_t id[128]);

/* ---- synthetic-weight generator, host mirror (for checkers) ---------------------------- */
/* dst[j] = element (first + j) of a tensor with the given seed/distribution; identical to
 * what l2b_create_synthetic puts on the device.                                            */
void l2b_synth_fill_host(float *dst, uint64_t first, uint64_t count, uint64_t tensor_seed,
                         double mean, double sigma, float lo, float hi);
/* Whole payload in checkpoint order (src/main.zig:85-112).                                 */
int32_t l2b_synth_checkpoint_host(const l2b_config *cfg, uint64_t seed, float *data,
                                  uint64_t n_floats);
uint64_t l2b_checkpoint_floats(const l2b_config *cfg);

/* ---- single ops with HOST buffers (unit-test surface) ---------------------------------- */
/* Each runs the same device code the hot path uses, on cuda:`device`, so the reference's
 * own unit tests (src/main.zig:1078-1150) can be replayed against the GPU.                 */
/* matmul (src/main.zig:485-498): xout(d) = W(d,n) . x(n)                                   */
int32_t l2b_op_matmul(int32_t device, float *xout, const float *x, const float *w, int32_t d,
                      int32_t n);
/* The fused pieces of the hot path in isolation: xout(d) = W(d,n) . rmsnorm(x, gamma) (gamma NULL
 * => W . x) through one GEMV kernel flavour (kernel: 0 = the library's own choice, 1 = latency
 * kernel, 2 = register-fed 8-row streaming kernel, 3 = TMA-ring streaming kernel).  With
 * resid_inout != NULL the result is instead accumulated into it (the residual add of :395/:422
 * in the epilogue) and xout is ignored.                                                    */
int32_t l2b_op_fused_matmul(int32_t device, float *xout, const float *x, const float *gamma,
                            const float *w, float *resid_inout, int32_t d, int32_t n,
                            int32_t kernel);
/* rmsnorm (:432-468)                                                                       */
int32_t l2b_op_rmsnorm(int32_t device, float *o, const float *x, const float *w, int32_t n);
/* softmax (:687-706), in place                                                             */
int32_t l2b_op_softmax(int32_t device, float *x, int32_t n);
/* vector_weighted_sum_rows (:657-685)                                                      */
int32_t l2b_op_weighted_sum_rows(int32_t device, float *xout, int32_t out_len, const float *rows,
                                 int32_t row_stride, const float *weights, int32_t n_weights);
/* One attention head over a KV cache slice (:361-389): q(head_size), keys/values are
 * (n_pos, kv_stride) row-major with the head's slice starting at column 0.                 */
int32_t l2b_op_attention_head(int32_t device, float *out, const float *q, const float *keys,
                              const float *values, int32_t head_size, int32_t kv_stride,
                              int32_t n_pos);

/* Sampler preparation alone (:1005-1008, :761-768) on n host logits, in place (see
 * l2b_forward_sample); *n_cand = number that passed the filter (-1 when top_p is 0 or 1).   */
int32_t l2b_op_sample_prep(int32_t device, float *logits_inout, int32_t n, float temperature,
                           float top_p, l2b_prob_index *cand, int32_t cand_cap, int32_t *n_cand);

#ifdef __cplusplus
}
#endif
#endif /* LLAMA2_B200_H */
