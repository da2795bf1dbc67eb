/*
 * qwen3_cuda.h -- C ABI of libqwen3cuda, the B200 (sm_100a) drop-in for qwen3-rs's quantized
 * forward pass.
 *
 * This is the boundary a Rust `qwen3-cuda` crate binds with `extern "C"` (see INTEGRATION.md)
 * to implement qwen3-inference's
 *
 *     pub trait Transformer {                                  // models/mod.rs:13-18
 *         fn forward(&mut self, token: usize, pos: usize) -> &[f32];
 *         fn get_config(&self) -> &ModelConfig;
 *     }
 *
 * and `TransformerBuilder::new(path).with_ctx_length(opt).build()` (models/mod.rs:40-74).
 * Plain pointers and sizes only; no exceptions cross the boundary.  Every entry point returns
 * 0 on success and a negative Q3_E* code on failure, with a message in q3_last_error().
 * A handle is owned by one caller thread at a time (the reference takes `&mut self`).
 * All file:line citations are relative to the reference repository root.
 */
#ifndef QWEN3_CUDA_H
#define QWEN3_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Q3_OK 0
#define Q3_EINVAL (-1)   /* bad argument (reference: panic on slice index / assert)        */
#define Q3_EIO (-2)      /* cannot open / map the checkpoint (models/mod.rs:56-59)          */
#define Q3_EFORMAT (-3)  /* bad magic / version / dims / short file (configuration.rs:116-146, utils.rs:21-26) */
#define Q3_ECUDA (-4)    /* CUDA runtime error                                              */
#define Q3_EUNSUPPORTED (-5) /* shape outside what the kernels cover (e.g. head_dim != 128) */
#define Q3_ECOMM (-6)    /* tensor-parallel communicator error                              */

/* POD mirror of ModelConfig (configuration.rs:18-30), same field meaning.  seq_len already has
 * the context-length override applied (models/mod.rs:65-67). */
typedef struct q3_config {
    int32_t architecture_id;
    int32_t dim;
    int32_t hidden_dim;
    int32_t n_layers;
    int32_t n_heads;
    int32_t n_kv_heads;
    int32_t head_dim;
    int32_t seq_len;
    int32_t vocab_size;
    int32_t group_size;
    int32_t shared_classifier;
} q3_config;

typedef struct q3_handle q3_handle;

/* ---- construction: TransformerBuilder (models/mod.rs:40-74) --------------------------------
 * Opens and validates the checkpoint (configuration.rs:77-146), uploads it once to HBM
 * (re-laid-out for the kernels), zero-fills the device KV cache (qwen3.rs:439-440) and uploads
 * the host-computed RoPE table (layers.rs:161-171).  ctx_len <= 0 keeps the file's seq_len.
 * device: CUDA ordinal. */
int q3_create(const char *checkpoint_path, int ctx_len, int device, q3_handle **out);

/* Tensor-parallel member: rank `tp_rank` of `tp_size` (one process per GPU).  Attention heads
 * and FFN columns are sharded (SURVEY.md §8e); the exchange after o_proj / down_proj runs over
 * NVLink peer memory.  After creating every rank call q3_tp_export / q3_tp_connect. */
int q3_create_tp(const char *checkpoint_path, int ctx_len, int device, int tp_rank, int tp_size,
                 q3_handle **out);
/* Size in bytes of the opaque per-rank blob (CUDA IPC handles of the exchange buffers). */
size_t q3_tp_blob_size(void);
int q3_tp_export(q3_handle *h, void *blob_out);
/* blobs: tp_size blobs, rank-major (all-gathered by the host, e.g. torch.distributed). */
int q3_tp_connect(q3_handle *h, const void *blobs);

/* Tensor parallel: by default q3_forward(logits_host != NULL) returns the full-vocabulary logits on EVERY rank (each
 * rank pushes its vocabulary shard to all peers).  With a logits root only that rank may ask for logits; the others call
 * q3_forward(..., NULL) / q3_forward_argmax for the same step and push their shard to the root alone.  root < 0 restores
 * the default.  Must be set identically on every rank. */
int q3_tp_set_logits_root(q3_handle *h, int root);

void q3_destroy(q3_handle *h);

/* ---- Transformer::get_config (models/mod.rs:17) ------------------------------------------- */
const q3_config *q3_get_config(const q3_handle *h);

/* ---- Transformer::forward (models/mod.rs:15, qwen3.rs:62-79) -------------------------------
 * Runs one decode step on the device and copies the vocab_size logits to logits_host (the
 * reference returns a borrow of its own logits that the caller copies, generation.rs:159-160).
 * logits_host == NULL leaves them on the device (see q3_logits_device).
 * token >= vocab_size or pos >= seq_len -> Q3_EINVAL (the reference panics). */
int q3_forward(q3_handle *h, int token, int pos, float *logits_host);

/* Extension (SURVEY.md §8f-1): forward + device-side greedy argmax with the reference's
 * tie rule (sampler.rs:57-59: last index among equal maxima).  Only 4 bytes cross PCIe. */
int q3_forward_argmax(q3_handle *h, int token, int pos, int *next_token);

/* Extension: n greedy steps entirely on the device (token feedback stays in HBM); tokens_out
 * receives the n sampled tokens.  Equivalent to n q3_forward_argmax calls starting at
 * (first_token, pos0). */
int q3_decode_greedy(q3_handle *h, int first_token, int pos0, int n, int *tokens_out);

/* Extension (SURVEY.md §8f-1, second half): the reference's Sampler (sampler.rs) on the device.
 * q3_sampler_set = Sampler::new(vocab, temperature, topp, rng_seed) (:30-41; the same argument checks, Q3_EINVAL instead
 * of the asserts).  q3_forward_sample = forward + Sampler::sample (:116-136): temperature 0 -> argmax; otherwise
 * temperature, softmax, xorshift64* coin, multinomial or top-p -- the same RNG stream and the same decisions as the
 * reference (order-sensitive sums are left folds, exp is glibc's; equal-probability candidates are taken in index
 * order, which the reference's unstable sort leaves unspecified).  Only the token crosses PCIe.
 * q3_decode_sample: n sampled steps entirely on the device.  q3_sampler_skip advances the RNG by n draws (the reference's
 * chat loop samples and discards once per prompt token, generation.rs:116-122; no-op when greedy).  q3_sampler_state
 * reads the RNG state back (Sampler::rng_state).  Under tensor parallelism every rank must be given the same seed. */
int q3_sampler_set(q3_handle *h, float temperature, float topp, unsigned long long rng_seed);
int q3_sampler_state(q3_handle *h, unsigned long long *rng_state_out);
int q3_sampler_skip(q3_handle *h, int n_draws);
int q3_forward_sample(q3_handle *h, int token, int pos, int *next_token);
int q3_decode_sample(q3_handle *h, int first_token, int pos0, int n, int *tokens_out);

/* Extension (SURVEY.md §8f-2): batched prefill of n tokens at positions pos0..pos0+n-1.  Leaves
 * the KV cache as n sequential forwards would (within float tolerance) and returns the logits
 * of the last token (NULL to skip). */
int q3_prefill(q3_handle *h, const int *tokens, int n, int pos0, float *last_logits_host);

/* Timing helper: one batched prefill of n tokens (after an untimed warm-up pass), CUDA events on the
 * launch stream, inputs resident; milliseconds. */
int q3_bench_prefill(q3_handle *h, const int *tokens, int n, int pos0, float *ms_out);

/* Extension: score n tokens at positions pos0..pos0+n-1 in one batched pass.
 * Leaves the KV cache exactly as q3_prefill(h, tokens, n, pos0, NULL) does.
 * For every i in [0, n), with logits_i = the logits after tokens[0..i] at position pos0+i:
 *   logprobs_out[i] = log softmax(logits_i)[targets[i]]   (natural log, f32; targets: n ids, required iff logprobs_out)
 *   argmax_out[i]   = argmax(logits_i), last index among equal maxima (sampler.rs:57-59, as q3_forward_argmax)
 * At least one of logprobs_out / argmax_out must be non-NULL.  q3_logits_device() is unspecified afterwards.
 * A target is scored at its own position, so a long text can be scored in pieces: the target of a piece's last position is
 * the first token of the next piece.  Every argument is checked before any device work (Q3_EINVAL; Q3_ECOMM for an
 * unconnected tensor-parallel handle): on an error nothing is written.  Fast mode runs the batched prefill, then the final
 * norm, the lm_head on the tensor cores and the reduction on every row; exact mode (or a shape without the batched path)
 * runs n q3_forward steps and reduces the reference's own logits.  Under tensor parallelism every rank runs the full lm_head
 * and returns the full results; there the batched path is required (Q3_EUNSUPPORTED otherwise). */
int q3_score(q3_handle *h, const int *tokens, int n, int pos0, const int *targets, float *logprobs_out, int *argmax_out);

/* Extension: q3_score plus the k most likely tokens at every position, 1 <= k <= min(Q3_TOPK_MAX, vocab_size).
 *   topk_ids_out[i*k + j]      = the j-th largest entry of logits_i: descending value, among equal values the larger index
 *                                first (so topk_ids_out[i*k] == argmax_out[i])
 *   topk_logprobs_out[i*k + j] = log softmax(logits_i)[topk_ids_out[i*k + j]]; bit-identical to q3_score's logprobs_out[i]
 *                                where that id is targets[i]
 * Both are required; targets / logprobs_out / argmax_out are optional, as in q3_score, and bit-identical to its outputs.
 * Same checks, cache effect, paths and tensor-parallel behaviour as q3_score.  The [seq_len][k] result buffers are allocated
 * on the first call and grow with k. */
#define Q3_TOPK_MAX 64
int q3_score_topk(q3_handle *h, const int *tokens, int n, int pos0, int k, int *topk_ids_out, float *topk_logprobs_out,
                  const int *targets, float *logprobs_out, int *argmax_out);

/* Zero the KV cache (a freshly built reference transformer, qwen3.rs:439-440). */
int q3_reset(q3_handle *h);

/* Device pointer to the logits of the last forward (vocab_size f32, valid until the next call). */
const float *q3_logits_device(const q3_handle *h);

/* The handle's own page-locked host buffer (vocab_size f32).  Passed as `logits_host` to q3_forward / q3_prefill, the logits are
 * DMA-ed straight into it and no second host copy is made -- the reference's `forward` returns a borrow of the transformer's own
 * logits buffer in the same way (models/qwen3.rs:78); valid until the next call on this handle. */
float *q3_logits_host(q3_handle *h);

/* Copy KV cache rows [pos0, pos0+n) of one layer to the host, layout [n][n_kv_heads*head_dim]
 * (the reference's cache layout, layers.rs:329-331), or overwrite them from the host.  A tensor-parallel handle holds
 * only its own kv heads: rows are [n][(n_kv_heads / tp_size) * head_dim], heads tp_rank * n_kv_heads / tp_size ... */
int q3_kv_read(q3_handle *h, int layer, int pos0, int n, float *k_host, float *v_host);
int q3_kv_write(q3_handle *h, int layer, int pos0, int n, const float *k_host, const float *v_host);

/* Run layers [layer0, layer1) of one decode step on a caller-supplied residual stream x
 * (dim f32, host), in place -- the production kernels, teacher-forced for layer-level parity
 * tests.  With run_head != 0 also final norm + lm_head into logits_host. */
int q3_forward_layers(q3_handle *h, int pos, int layer0, int layer1, float *x_host, int run_head,
                      float *logits_host);

/* Which execution path q3_forward uses: 0 = multi-kernel CUDA graph, 1 = persistent
 * single-launch decode kernel.  Default: the fastest available. */
int q3_set_decode_path(q3_handle *h, int path);

/* Reference-order mode.  on != 0: every float reduction on the path (RMSNorm sum of squares,
 * QK-norm, GEMV group fold, attention scores / softmax denominator / value mix) is evaluated in
 * the reference's left-fold order and exp() is glibc's expf algorithm, so -- unlike the default
 * fast mode, which differs in summation order only -- logits are bit-identical to the
 * reference's.  Same kernels otherwise; slower (serial sums).  Used to demonstrate exact parity. */
int q3_set_exact(q3_handle *h, int on);
/* One reduction at a time (attribution of where the fast mode's int8 flips come from): bit 0 RMSNorm sum of squares,
 * bit 1 GEMV group fold, bit 2 QK-norm sum of squares, bit 3 attention (score dots, softmax with glibc expf, value mix),
 * bit 4 glibc expf in SwiGLU.  mask 31 == q3_set_exact(h, 1), mask 0 == fast mode. */
int q3_set_exact_mask(q3_handle *h, int mask);

/* Timing helper for benchmarks: runs `steps` decode steps at positions pos0.. (greedy token
 * feedback on the device) with inputs already resident, timed with CUDA events on the launch
 * stream; returns total milliseconds. */
int q3_bench_decode(q3_handle *h, int first_token, int pos0, int steps, float *ms_out);
/* Roofline helper: times ONE kernel family in isolation with CUDA events on the launch stream.
 * kind: 0 qkv GEMV, 1 o_proj GEMV, 2 gate/up GEMV (+SwiGLU), 3 down GEMV, 4 lm_head GEMV,
 * 5 decode attention at position `pos`.  Each rep launches the kernel once per layer (distinct
 * weights every launch, so the working set is far larger than L2).  Outputs: total milliseconds,
 * number of launches, algorithmic bytes per launch (weights + scales, or K/V rows read). */
int q3_bench_kernel(q3_handle *h, int kind, int pos, int reps, float *ms_out, int *launches_out,
                    double *bytes_per_launch_out);
/* Developer aid: one decode step of the persistent kernel with per-CTA tagged clock64 stamps (prof_mark in
 * csrc/q3_mega.cuh).  out: [n_rows][n_events] u64 words of (clock64 << 8 | tag); n_rows = 3 * q3_num_sms(h) (consumer
 * thread 0, producer 0, first lane of consumer group 1 of every CTA), the last word of a row is its event count.
 * out_words is the capacity of `out` in 64-bit words: too small -> Q3_EINVAL, nothing is written.  out == NULL with
 * out_words == 0 only returns the two sizes.  token / pos are validated like q3_forward. */
int q3_debug_profile(q3_handle *h, int token, int pos, unsigned long long *out, size_t out_words, int *n_rows_out,
                     int *n_events_out);
/* Number of SMs (= CTAs of the persistent kernel) of the handle's device. */
int q3_num_sms(const q3_handle *h);
/* Test hook: set the number of flagged exchanges issued so far (the persistent kernel's epochs are this counter
 * mod 2^32 - 1, plus 1), e.g. just below the wrap.  Every tensor-parallel rank must be given the same value. */
int q3_debug_set_epoch(q3_handle *h, unsigned long long exchanges_issued);
/* Number of kernel launches one decode step issues on the current path. */
int q3_launches_per_step(const q3_handle *h);

/* ---- operator-level entry points (host buffers in/out; used by the parity tests) -----------
 * Each runs the same device code the forward pass uses. */
/* tensor.rs:91-119 quantize */
int q3_op_quantize(int device, const float *x, int n, int gs, int8_t *q_out, float *s_out);
/* tensor.rs:23-62 matmul: out[d] from x (int8[n] + f32[n/gs]) and row-major w (int8[d*n] +
 * f32[d*n/gs]).  group_dots_out (optional, int32[d*(n/gs)]) receives the per-group integer
 * dot products the kernel accumulated.  exact != 0: reference-order group fold (bit-identical
 * f32 result), see q3_set_exact. */
int q3_op_matmul(int device, const int8_t *xq, const float *xs, const int8_t *wq, const float *ws,
                 int n, int d, int gs, int exact, float *out, int32_t *group_dots_out);
/* glibc expf restated on the device (exact mode's exp); x, out: n f32. */
int q3_op_expf(int device, const float *x, int n, float *out);
/* T-token group-scaled int8 GEMM on the tensor cores (tcgen05.mma.kind::i8, TMEM accumulators, TMA
 * operands): out[T][N] = per-token tensor.rs:23-62 matmul of x (int8[T][K] + f32[T][K/gs]) with
 * row-major w (int8[N][K] + f32[N][K/gs]).  N, K multiples of 128.  The int32 group dots are exact either way;
 * exact == 1: the f32 group terms are unfused and added in group order -- bit-identical to the per-token GEMV in exact
 * mode; exact == 0: the drain q3_prefill runs (fused multiply-add per group, same order of groups).  Any other value of
 * exact is Q3_EINVAL. */
int q3_op_gemm_q8(int device, const int8_t *xq, const float *xs, const int8_t *wq, const float *ws,
                  int T, int N, int K, int gs, int exact, float *out);
/* layers.rs:374-419 for T query tokens at once (the batched prefill's causal attention): q [T][n_heads*128] after QK-norm
 * and RoPE, k / v [pos0+T][n_kv*128] cache rows, out [T][n_heads*128].  The tensor-core kernel q3_prefill runs
 * (mma.sync m16n8k16 on an FP16 hi / lo split of the operands, f32 accumulation). */
int q3_op_prefill_attention(int device, const float *q, const float *k, const float *v, int T, int pos0, int n_heads,
                            int n_kv, float *out);
/* Timing helper: the tensor-core GEMM alone on device-resident pseudo-random operands (CUDA events, best of reps,
 * milliseconds per launch).  mode 0 / 1 as `exact` above; any other mode is Q3_EINVAL. */
int q3_bench_gemm_q8(int device, int T, int N, int K, int gs, int mode, int reps, float *ms_out);
/* sampler.rs:116-136 Sampler::sample with temperature > 0 on host-supplied logits (n f32): one draw on the device;
 * *rng_state is Sampler::rng_state before the call and after it. */
int q3_op_sample(int device, const float *logits, int n, float temperature, float topp, unsigned long long *rng_state,
                 int *token_out);
/* The reduction q3_score runs, on host-supplied logits [rows][n] (operator-level parity tests). */
int q3_op_logprobs(int device, const float *logits, int rows, int n, const int *targets, float *logprobs_out, int *argmax_out);
/* The reduction q3_score_topk runs, on host-supplied logits [rows][n]: ids_out / lps_out [rows][k] (required), 1 <= k <=
 * min(Q3_TOPK_MAX, n); logprobs_out (needs targets) and argmax_out optional, as in q3_op_logprobs. */
int q3_op_topk_logprobs(int device, const float *logits, int rows, int n, int k, const int *targets, int *ids_out, float *lps_out,
                        float *logprobs_out, int *argmax_out);
/* layers.rs:109-119 RMSNorm::forward */
int q3_op_rmsnorm(int device, const float *x, const float *w, int n, float *out);
/* qwen3-export model_exporter.rs:104-161 quantize_q80 on the device (SURVEY.md §8f-3). */
int q3_op_quantize_q80(int device, const float *w, size_t n, int gs, int8_t *q_out, float *s_out);
/* The same kernel on DEVICE buffers (w_dev: n f32, q_dev: n int8, s_dev: n/gs f32, all on `device`): how the synthetic
 * multi-GB bench / test checkpoints are quantised. */
int q3_op_quantize_q80_dev(int device, const float *w_dev, size_t n, int gs, int8_t *q_dev, float *s_dev);

const char *q3_last_error(void);
const char *q3_version(void);

#ifdef __cplusplus
}
#endif
#endif /* QWEN3_CUDA_H */
