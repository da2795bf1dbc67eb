// q3_engine.cu -- host side of libqwen3cuda: checkpoint loader, HBM layout, decode graph and
// the extern "C" API declared in include/qwen3_cuda.h.
//
// Mirrors the reference's construction path: TransformerBuilder::build (models/mod.rs:55-73) ->
// read_config (configuration.rs:77-146) -> load_weights (qwen3.rs:199-277) ->
// TransformerBlockBuffers::new (qwen3.rs:412-445), then Qwen3Transformer::forward (qwen3.rs:62-79).
#include "../../include/qwen3_cuda.h"
#include "q3_kernels.cuh"
#include "q3_mega.cuh"
#include "q3_prefill.cuh"
#include "q3_sampler.cuh"
#include <cudaTypedefs.h>

#include <cuda_runtime.h>
#include <fcntl.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <string>
#include <vector>

using namespace q3;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return fail(Q3_ECUDA, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, __LINE__, \
                        cudaGetErrorString(e_));                                                        \
    } while (0)

extern "C" const char *q3_last_error(void) { return g_err; }

extern "C" const char *q3_version(void) { return "qwen3cuda 0.1 (sm_100a)"; }

// Milliseconds of GPU time from an event recorded on `s` before work() to one recorded after it, once the stream's earlier work
// has finished.  The events are destroyed on every path.
template <class F>
static int time_events(cudaStream_t s, float *ms, F &&work) {
    struct Events {
        cudaEvent_t e[2] = {nullptr, nullptr};
        ~Events() {
            for (cudaEvent_t x : e)
                if (x) cudaEventDestroy(x);
        }
    } ev;
    CK(cudaEventCreate(&ev.e[0]));
    CK(cudaEventCreate(&ev.e[1]));
    CK(cudaStreamSynchronize(s));
    CK(cudaEventRecord(ev.e[0], s));
    if (int rc = work()) return rc;
    CK(cudaEventRecord(ev.e[1], s));
    CK(cudaEventSynchronize(ev.e[1]));
    CK(cudaGetLastError());
    CK(cudaEventElapsedTime(ms, ev.e[0], ev.e[1]));
    return 0;
}

// ------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------
struct DevQT { // device QuantizedTensor: row-major int8 [rows][K] + f32 scales [rows][K/gs]
    int8_t *q = nullptr;
    float *s = nullptr;
    int rows = 0, K = 0;
    float *sT = nullptr;      // prefill: scales group-major [K/gs][rows]
    CUtensorMap map{};        // prefill: TMA map over q, box 128 rows x 128 B, 128B swizzle
    bool has_map = false;
};

struct LayerDev {
    DevQT qkv; // rows: [AH_l q | KV_l k | KV_l v]            (layers.rs:334-336 fused)
    DevQT wo;  // [dim][AH_l]
    DevQT w13; // rows interleaved (gate_j, up_j), j < H_l      (layers.rs:468-469 fused)
    DevQT w2;  // [dim][H_l]
    float *rms_att = nullptr, *rms_ffn = nullptr, *q_ln = nullptr, *k_ln = nullptr;
};

struct q3_handle {
    q3_config cfg{};
    int device = 0;
    int tp_rank = 0, tp_size = 1;
    int n_heads_l = 0, n_kv_l = 0, AH_l = 0, KV_l = 0, H_l = 0, kv_mul = 1;
    int num_sms = 148;
    std::vector<LayerDev> layers;
    DevQT embed, wcls;
    float *rms_final = nullptr;
    float *rope = nullptr; // [seq_len][64][2]
    // activations
    float *x = nullptr, *xb = nullptr, *q = nullptr, *hb = nullptr, *logits = nullptr, *attn_part = nullptr;
    unsigned *att_cnt = nullptr; // persistent kernel: per (layer, kv head) arrival counters of the attention splits
    int8_t *xq = nullptr, *hq = nullptr;
    float *xs = nullptr, *hs = nullptr;
    float *kc = nullptr, *vc = nullptr; // [L][seq_len][KV_l]
    int *d_tokpos = nullptr;            // [0]=token [1]=pos [2]=argmax out [3]=history idx
    int *d_history = nullptr;
    int history_cap = 0;
    float *h_logits = nullptr; // pinned
    int *h_small = nullptr;    // pinned scratch
    cudaStream_t stream = nullptr;
    cudaGraphExec_t g_fwd[32] = {}, g_greedy[32] = {}; // [exact mask]
    // Reference-order mask (bit-level parity mode; q3_set_exact = all bits, q3_set_exact_mask = per reduction, for the
    // attribution of int8 flips): 1 RMSNorm sum of squares, 2 GEMV group fold, 4 QK-norm sum of squares,
    // 8 attention (score dots, softmax with glibc expf, value mix), 16 glibc expf in SwiGLU
    int exact = 0;
    float *att = nullptr;   // exact mode scratch [n_heads_l][seq_len] (the reference's `att`)
    int decode_path = 0;    // 0 = multi-kernel CUDA graph, 1 = persistent megakernel
    int launches_per_step = 0, graph_launches_per_step = 0;
    // megakernel state
    bool mega_ok = false;
    std::string mega_why;
    MegaArgs margs{};
    unsigned long long bar_base = 0, xbar_base = 0;
    int *d_status = nullptr;  // device abort flag raised by a timed-out wait inside the kernel
    unsigned long long *part_buf[2] = {nullptr, nullptr};            // TP landing zones [tp][dim] (inside xchg: peers write them)
    unsigned long long *zq = nullptr, *za = nullptr, *zh = nullptr, *zr[2] = {nullptr, nullptr}; // local (payload, epoch) zones
    int logits_root = -1;     // TP: >= 0 = only this rank receives the other ranks' vocabulary shards (q3_tp_set_logits_root)
    bool poisoned = false;    // a wait timed out under tensor parallelism: the ranks' epoch / barrier sequences may have diverged
    unsigned long long *d_best = nullptr, *d_bar = nullptr;
    unsigned int *d_flags = nullptr;
    // everything a TP peer writes into lives in ONE allocation (one CUDA IPC handle per rank):
    // [part o_proj | part down | argmax candidates | barrier flags | logits]
    uint8_t *xchg = nullptr;
    size_t xchg_bytes = 0, off_part[2] = {0, 0}, off_best = 0, off_flags = 0, off_logits = 0;
    // batched prefill under TP: two partial blocks [pf_tp_cap][dim] f32 + an arrival counter inside the exchange buffer
    size_t off_pf_part[2] = {0, 0}, off_pf_ctr = 0;
    int pf_tp_cap = 0;                     // tokens per prefill chunk under TP (longer prompts go through in chunks)
    PfPeers pf_peers[2]{};                 // peer views of the two partial blocks (+ counters), filled by q3_tp_connect
    unsigned long long pf_xbar_count = 0;  // cross-GPU prefill barriers passed so far (same sequence on every rank)
    bool tp_connected = false;
    std::vector<void *> peer_maps;
    size_t mega_smem = 0;
    unsigned long long ll_count = 0; // flagged exchanges issued so far (same sequence on every TP rank); epochs derive from it
    void *mega_fn = nullptr;
    // batched prefill (tcgen05 GEMM) state
    bool pf_ok = false;
    std::string pf_why;
    __half *pf_kvh = nullptr; // [4][pf_kvh_rows][KV_l] halves: this layer's K / V rows split into hi / lo (k_pf_split_kv)
    size_t pf_kvh_rows = 0;
    int pf_cap = 0;          // token capacity of the buffers below (multiple of 128)
    float *pf_x = nullptr, *pf_q = nullptr, *pf_att = nullptr, *pf_hb = nullptr, *pf_xsT = nullptr, *pf_hsT = nullptr;
    int8_t *pf_xq = nullptr, *pf_hq = nullptr;
    int *pf_tokens = nullptr;
    // q3_score, allocated on its first call: per-position targets / results [seq_len], the lm_head rows of one chunk
    // [sc_cap][vocab] f32 (grow-only, freed in q3_destroy)
    int *sc_targets = nullptr, *sc_argmax = nullptr;
    float *sc_lp = nullptr, *sc_logits = nullptr;
    int sc_cap = 0;
    bool sc_want_lp = false; // this call asked for log-probabilities (targets uploaded)
    // q3_score_topk, allocated on its first call: ids / log-probabilities [seq_len][tk_cap] (grow-only in k, freed in q3_destroy)
    int *tk_ids = nullptr;
    float *tk_lps = nullptr;
    int tk_cap = 0;
    int tk_k = 0; // k of this call; 0 in q3_score
    // device sampler (sampler.rs on the device, q3_sampler.cuh)
    float samp_temperature = 0.0f, samp_topp = 0.9f;
    unsigned long long *d_rng = nullptr, *d_keys = nullptr;
    float *d_probs = nullptr;
    size_t dev_bytes = 0;
    std::vector<void *> allocs;
};

static int dmalloc(q3_handle *h, void **p, size_t bytes) {
    CK(cudaMalloc(p, bytes ? bytes : 16));
    h->allocs.push_back(*p);
    h->dev_bytes += bytes;
    return 0;
}

// ------------------------------------------------------------------------------------------
// checkpoint (configuration.rs, utils.rs)
// ------------------------------------------------------------------------------------------
struct HostQT {
    const int8_t *q;
    const float *s;
};
struct Ckpt {
    uint8_t *map = nullptr;
    size_t len = 0, off = 0;
    q3_config cfg{};
    const float *rms_att, *rms_ffn, *rms_final, *q_ln, *k_ln;
    HostQT embed, wcls;
    std::vector<HostQT> wq, wk, wv, wo, w1, w2, w3;
    ~Ckpt() {
        if (map) munmap(map, len);
    }
    const void *take(size_t bytes) { // utils.rs:21-49
        if (off + bytes > len) return nullptr;
        const void *p = map + off;
        off += bytes;
        return p;
    }
};

static int open_ckpt(const char *path, int ctx_len, Ckpt &c) {
    int fd = open(path, O_RDONLY);
    if (fd < 0) return fail(Q3_EIO, "Failed to open checkpoint: %s", path);
    struct stat st;
    fstat(fd, &st);
    c.len = (size_t)st.st_size;
    void *m = mmap(nullptr, c.len ? c.len : 1, PROT_READ, MAP_PRIVATE, fd, 0);
    close(fd);
    if (m == MAP_FAILED) return fail(Q3_EIO, "Failed to create memory mapping");
    c.map = (uint8_t *)m;
    const int32_t *hd = (const int32_t *)c.take(13 * 4);
    if (!hd) return fail(Q3_EFORMAT, "Insufficient data for config: need 52 bytes, got %zu", c.len);
    if (hd[0] != 0x616a6331)
        return fail(Q3_EFORMAT, "Invalid checkpoint magic number: expected 0x616a6331, got %#x", hd[0]);
    if (hd[1] != 1) return fail(Q3_EFORMAT, "Unsupported checkpoint version: expected 1, got %d", hd[1]);
    const char *names[8] = {"architecture_id", "dim", "n_layers", "n_heads", "n_kv_heads", "vocab_size", "seq_len", "head_dim"};
    int32_t vals[8] = {hd[2], hd[3], hd[5], hd[6], hd[7], hd[8], hd[9], hd[10]};
    for (int i = 0; i < 8; i++)
        if (vals[i] <= 0) return fail(Q3_EFORMAT, "Invalid %s: must be positive, got %d", names[i], vals[i]);
    if (!c.take(256 - 52)) return fail(Q3_EFORMAT, "Cannot skip %d bytes: insufficient data", 256 - 52);
    q3_config &cf = c.cfg;
    cf.architecture_id = hd[2]; cf.dim = hd[3]; cf.hidden_dim = hd[4]; cf.n_layers = hd[5];
    cf.n_heads = hd[6]; cf.n_kv_heads = hd[7]; cf.vocab_size = hd[8]; cf.seq_len = hd[9];
    cf.head_dim = hd[10]; cf.shared_classifier = hd[11] != 0; cf.group_size = hd[12];
    if (ctx_len > 0 && ctx_len < cf.seq_len) cf.seq_len = ctx_len; // models/mod.rs:65-67
    if (cf.architecture_id != 1) return fail(Q3_EFORMAT, "Unknown architecture_id: %d", cf.architecture_id);
    if (cf.hidden_dim <= 0 || cf.group_size <= 0) return fail(Q3_EFORMAT, "Invalid hidden_dim/group_size");

    const int L = cf.n_layers, dim = cf.dim, hdm = cf.head_dim, gs = cf.group_size;
    const size_t AH = (size_t)cf.n_heads * hdm, KV = (size_t)cf.n_kv_heads * hdm, H = cf.hidden_dim, V = cf.vocab_size;
#define TAKE_F32(dst, n, what)                                                         \
    if (!((dst) = (const float *)c.take((size_t)(n) * 4)))                             \
        return fail(Q3_EFORMAT, "Failed to read %s: Insufficient data", what);
    TAKE_F32(c.rms_att, (size_t)L * dim, "attention normalization weights");
    TAKE_F32(c.rms_ffn, (size_t)L * dim, "FFN normalization weights");
    TAKE_F32(c.rms_final, dim, "final normalization weights");
    TAKE_F32(c.q_ln, (size_t)L * hdm, "query layer norm weights");
    TAKE_F32(c.k_ln, (size_t)L * hdm, "key layer norm weights");
    auto take_qts = [&](std::vector<HostQT> &v, int n, size_t size_each, const char *what) -> int {
        v.resize(n);
        for (int i = 0; i < n; i++) { // models/mod.rs:89-108
            v[i].q = (const int8_t *)c.take(size_each);
            v[i].s = (const float *)c.take(size_each / gs * 4);
            if (!v[i].q || !v[i].s)
                return fail(Q3_EFORMAT, "Failed to read quantized tensor %d data (%s): Insufficient data", i, what);
        }
        return 0;
    };
    std::vector<HostQT> one;
    int rc;
    if ((rc = take_qts(one, 1, V * dim, "token embedding"))) return rc;
    c.embed = one[0];
    if ((rc = take_qts(c.wq, L, (size_t)dim * AH, "wq"))) return rc;
    if ((rc = take_qts(c.wk, L, (size_t)dim * KV, "wk"))) return rc;
    if ((rc = take_qts(c.wv, L, (size_t)dim * KV, "wv"))) return rc;
    if ((rc = take_qts(c.wo, L, AH * dim, "wo"))) return rc;
    if ((rc = take_qts(c.w1, L, (size_t)dim * H, "w1"))) return rc;
    if ((rc = take_qts(c.w2, L, H * dim, "w2"))) return rc;
    if ((rc = take_qts(c.w3, L, (size_t)dim * H, "w3"))) return rc;
    if (cf.shared_classifier) c.wcls = c.embed;
    else {
        if ((rc = take_qts(one, 1, (size_t)dim * V, "classifier"))) return rc;
        c.wcls = one[0];
    }
    return 0;
}

// ------------------------------------------------------------------------------------------
// upload helpers
// ------------------------------------------------------------------------------------------
struct Stager { // pinned staging buffer for re-laid-out tensors
    uint8_t *buf = nullptr;
    size_t cap = 0;
    ~Stager() {
        if (buf) cudaFreeHost(buf);
    }
    int ensure(size_t n) {
        if (n <= cap) return 0;
        if (buf) cudaFreeHost(buf);
        buf = nullptr;
        cap = 0;
        CK(cudaMallocHost((void **)&buf, n));
        cap = n;
        return 0;
    }
};

// Allocate a device tensor of `rows` x K and fill it from row pieces: piece i copies
// rows[i] rows starting at source row src_row0[i] of src[i], columns [col0, col0+K) of a
// source matrix with srcK columns (col slicing = row-parallel TP shard of Wo / W2).
struct RowPiece {
    HostQT src;
    int src_row0, nrows, srcK;
};
static int upload_rows(q3_handle *h, Stager &st, DevQT &dst, const std::vector<RowPiece> &pieces, int K, int col0,
                       int gs, bool interleave2 = false) {
    int rows = 0;
    for (auto &p : pieces) rows += p.nrows;
    dst.rows = rows;
    dst.K = K;
    const int ng = K / gs;
    size_t qbytes = (size_t)rows * K, sbytes = (size_t)rows * ng * 4;
    int rc;
    if ((rc = dmalloc(h, (void **)&dst.q, qbytes))) return rc;
    if ((rc = dmalloc(h, (void **)&dst.s, sbytes))) return rc;
    if ((rc = st.ensure(qbytes + sbytes))) return rc;
    int8_t *hq = (int8_t *)st.buf;
    float *hs = (float *)(st.buf + qbytes);
    if (interleave2) { // two pieces of equal size, rows alternate (gate_j, up_j)
        const RowPiece &a = pieces[0], &b = pieces[1];
        for (int j = 0; j < a.nrows; j++) {
            const RowPiece *pp[2] = {&a, &b};
            for (int t = 0; t < 2; t++) {
                size_t sr = (size_t)pp[t]->src_row0 + j;
                memcpy(hq + (size_t)(2 * j + t) * K, pp[t]->src.q + sr * pp[t]->srcK + col0, K);
                memcpy(hs + (size_t)(2 * j + t) * ng, pp[t]->src.s + sr * (pp[t]->srcK / gs) + col0 / gs, (size_t)ng * 4);
            }
        }
    } else {
        size_t r = 0;
        for (auto &p : pieces) {
            if (p.srcK == K && col0 == 0) {
                memcpy(hq + r * K, p.src.q + (size_t)p.src_row0 * K, (size_t)p.nrows * K);
                memcpy(hs + r * ng, p.src.s + (size_t)p.src_row0 * ng, (size_t)p.nrows * ng * 4);
            } else {
                for (int j = 0; j < p.nrows; j++) {
                    size_t sr = (size_t)p.src_row0 + j;
                    memcpy(hq + (r + j) * K, p.src.q + sr * p.srcK + col0, K);
                    memcpy(hs + (r + j) * ng, p.src.s + sr * (p.srcK / gs) + col0 / gs, (size_t)ng * 4);
                }
            }
            r += p.nrows;
        }
    }
    CK(cudaMemcpy(dst.q, hq, qbytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dst.s, hs, sbytes, cudaMemcpyHostToDevice));
    return 0;
}
static int upload_f32(q3_handle *h, float **dst, const float *src, size_t n) {
    int rc;
    if ((rc = dmalloc(h, (void **)dst, n * 4))) return rc;
    CK(cudaMemcpy(*dst, src, n * 4, cudaMemcpyHostToDevice));
    return 0;
}

// ------------------------------------------------------------------------------------------
// kernel launch sequence (qwen3.rs:62-79, 131-176)
// ------------------------------------------------------------------------------------------
#define GS_DISPATCH(gs, CALL)                \
    switch (gs) {                            \
    case 32: { constexpr int GS = 32; CALL; } break;   \
    case 64: { constexpr int GS = 64; CALL; } break;   \
    case 128: { constexpr int GS = 128; CALL; } break; \
    default: break;                          \
    }
// GQA factor (query heads per kv head); create_impl admits only these four
#define KV_DISPATCH(kv_mul, CALL)                          \
    switch (kv_mul) {                                      \
    case 1: { constexpr int KVM = 1; CALL; } break;        \
    case 2: { constexpr int KVM = 2; CALL; } break;        \
    case 4: { constexpr int KVM = 4; CALL; } break;        \
    case 8: { constexpr int KVM = 8; CALL; } break;        \
    default: break;                                        \
    }

template <int GS, int EPI>
static void launch_gemv_t(int num_sms, int exact, GemvArgs a, cudaStream_t s) {
    int npairs = a.rows / 2;
    int grid = (npairs + 7) / 8;
    int cap = num_sms * 8;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    size_t smem = (size_t)a.K + (size_t)(a.K / GS) * 4;
    const bool expref = EPI == EPI_SWIGLU && (exact & 16);
    if (exact & 2) {
        smem += (size_t)16 * (a.K / GS) * 4; // [8 warps][2 rows][ng] terms
        if (expref) k_gemv<GS, EPI, true, true><<<grid, 256, smem, s>>>(a);
        else k_gemv<GS, EPI, true, false><<<grid, 256, smem, s>>>(a);
    } else {
        if (expref) k_gemv<GS, EPI, false, true><<<grid, 256, smem, s>>>(a);
        else k_gemv<GS, EPI, false, false><<<grid, 256, smem, s>>>(a);
    }
}
// exact: the reference-order mask (q3_handle::exact)
template <int EPI>
static void launch_gemv(int gs, int num_sms, int exact, const GemvArgs &a, cudaStream_t s) {
    GS_DISPATCH(gs, (launch_gemv_t<GS, EPI>(num_sms, exact, a, s)));
}

static int launch_norm_quant(int gs, int exact, const NormQuantArgs &a, cudaStream_t s) {
    if (exact & 1) {
        GS_DISPATCH(gs, (k_rmsnorm_quant<GS, true><<<1, 1024, (size_t)a.n * 4, s>>>(a)));
    } else {
        GS_DISPATCH(gs, (k_rmsnorm_quant<GS, false><<<1, 1024, 0, s>>>(a)));
    }
    return 1;
}

// split-K decode attention of one layer at position d_tokpos[1]: partials of ATTN_MAX_SPLITS CTAs per kv head into attn_part
static void launch_attn_partial(const q3_handle *h, const float *kc_l, const float *vc_l, cudaStream_t s) {
    dim3 ag(h->n_kv_l, ATTN_MAX_SPLITS);
    KV_DISPATCH(h->kv_mul, (k_attn_partial<KVM><<<ag, 128, 0, s>>>(h->q, kc_l, vc_l, h->attn_part, h->d_tokpos + 1, h->KV_l, h->n_heads_l)));
}

// One transformer block.  Returns the number of kernel launches.
static int launch_layer(q3_handle *h, int l, bool first_from_embed, cudaStream_t s) {
    const q3_config &c = h->cfg;
    const LayerDev &W = h->layers[l];
    const int gs = c.group_size, dim = c.dim, ns = h->num_sms, ex = h->exact;
    const int *d_token = h->d_tokpos, *d_pos = h->d_tokpos + 1;
    float *kc_l = h->kc + (size_t)l * c.seq_len * h->KV_l;
    float *vc_l = h->vc + (size_t)l * c.seq_len * h->KV_l;
    int n = 0;
    // attn_norm + quantize (qwen3.rs:134-136); layer 0 also gathers the embedding row (qwen3.rs:64)
    NormQuantArgs na{};
    na.x = h->x; na.w = W.rms_att; na.q = h->xq; na.s = h->xs; na.n = dim;
    if (first_from_embed) { na.embed_q = h->embed.q; na.embed_s = h->embed.s; na.token = d_token; }
    n += launch_norm_quant(gs, ex, na, s);
    // q, k, v projections (layers.rs:334-336)
    GemvArgs g{};
    g.wq = W.qkv.q; g.ws = W.qkv.s; g.xq = h->xq; g.xs = h->xs; g.K = dim; g.rows = W.qkv.rows;
    g.q = h->q; g.kc = kc_l; g.vc = vc_l; g.AH = h->AH_l; g.KV = h->KV_l; g.pos = d_pos;
    launch_gemv<EPI_QKV>(gs, ns, ex, g, s); n++;
    // QK-norm + RoPE (layers.rs:339-340)
    int nh = h->n_heads_l + h->n_kv_l;
    if (h->exact & 4)
        k_qknorm_rope<true><<<(nh + 3) / 4, 128, 0, s>>>(h->q, kc_l, W.q_ln, W.k_ln, h->rope, d_pos, h->n_heads_l, h->n_kv_l, h->KV_l);
    else
        k_qknorm_rope<false><<<(nh + 3) / 4, 128, 0, s>>>(h->q, kc_l, W.q_ln, W.k_ln, h->rope, d_pos, h->n_heads_l, h->n_kv_l, h->KV_l);
    n++;
    // attention (layers.rs:343) + quantize (qwen3.rs:152)
    if (h->exact & 8) {
        k_attn_ordered<<<h->n_heads_l, 128, 0, s>>>(h->q, kc_l, vc_l, h->att, h->xb, d_pos, h->KV_l, h->kv_mul, c.seq_len);
        int n4 = h->AH_l / 4, grid = (n4 + 255) / 256;
        GS_DISPATCH(gs, (k_quantize<GS><<<grid, 256, 0, s>>>(h->xb, h->AH_l, h->xq, h->xs)));
        n += 2;
    } else {
        launch_attn_partial(h, kc_l, vc_l, s);
        GS_DISPATCH(gs, (k_attn_combine_quant<GS><<<h->n_heads_l, 128, 0, s>>>(h->attn_part, d_pos, h->xb, h->xq, h->xs)));
        n += 2;
    }
    // o_proj + residual (qwen3.rs:153-156)
    GemvArgs o{};
    o.wq = W.wo.q; o.ws = W.wo.s; o.xq = h->xq; o.xs = h->xs; o.K = h->AH_l; o.rows = dim; o.out = h->x;
    launch_gemv<EPI_RESID>(gs, ns, ex, o, s); n++;
    // ffn_norm + quantize (qwen3.rs:159-161)
    NormQuantArgs nf{};
    nf.x = h->x; nf.w = W.rms_ffn; nf.q = h->xq; nf.s = h->xs; nf.n = dim;
    n += launch_norm_quant(gs, ex, nf, s);
    // gate/up + SwiGLU (layers.rs:468-475)
    GemvArgs gu{};
    gu.wq = W.w13.q; gu.ws = W.w13.s; gu.xq = h->xq; gu.xs = h->xs; gu.K = dim; gu.rows = W.w13.rows; gu.out = h->hb;
    launch_gemv<EPI_SWIGLU>(gs, ns, ex, gu, s); n++;
    // quantize(hb) (layers.rs:478)
    {
        int n4 = h->H_l / 4, grid = (n4 + 255) / 256;
        GS_DISPATCH(gs, (k_quantize<GS><<<grid, 256, 0, s>>>(h->hb, h->H_l, h->hq, h->hs)));
        n++;
    }
    // down + residual (layers.rs:479, qwen3.rs:175)
    GemvArgs dn{};
    dn.wq = W.w2.q; dn.ws = W.w2.s; dn.xq = h->hq; dn.xs = h->hs; dn.K = h->H_l; dn.rows = dim; dn.out = h->x;
    launch_gemv<EPI_RESID>(gs, ns, ex, dn, s); n++;
    return n;
}

// final norm (in place) + quantize + lm_head (qwen3.rs:72-76)
static int launch_head(q3_handle *h, cudaStream_t s) {
    const q3_config &c = h->cfg;
    NormQuantArgs na{};
    na.x = h->x; na.w = h->rms_final; na.q = h->xq; na.s = h->xs; na.n = c.dim; na.write_normed = 1;
    int n = launch_norm_quant(c.group_size, h->exact, na, s);
    GemvArgs g{};
    g.wq = h->wcls.q; g.ws = h->wcls.s; g.xq = h->xq; g.xs = h->xs; g.K = c.dim; g.rows = c.vocab_size; g.out = h->logits;
    launch_gemv<EPI_STORE>(c.group_size, h->num_sms, h->exact, g, s); n++;
    return n;
}

static int launch_argmax(q3_handle *h, bool feedback, cudaStream_t s) {
    int *tp = h->d_tokpos;
    k_argmax<<<1, 1024, 0, s>>>(h->logits, h->cfg.vocab_size, tp + 2, feedback ? tp : nullptr, feedback ? tp + 1 : nullptr,
                                feedback ? h->d_history : nullptr, tp + 3);
    return 1;
}

static int launch_step(q3_handle *h, bool argmax, bool feedback, cudaStream_t s) {
    int n = 0;
    for (int l = 0; l < h->cfg.n_layers; l++) n += launch_layer(h, l, l == 0, s);
    n += launch_head(h, s);
    if (argmax) n += launch_argmax(h, feedback, s);
    return n;
}

static int build_graphs(q3_handle *h) {
    const int ex = h->exact;
    for (int which = 0; which < 2; which++) {
        cudaGraphExec_t *slot = which ? &h->g_greedy[ex] : &h->g_fwd[ex];
        cudaGraph_t g;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        int n = launch_step(h, which == 1, which == 1, h->stream);
        cudaError_t e = cudaStreamEndCapture(h->stream, &g);
        if (e != cudaSuccess) return fail(Q3_ECUDA, "graph capture failed: %s", cudaGetErrorString(e));
        if (!*slot) CK(cudaGraphInstantiate(slot, g, 0));
        CK(cudaGraphDestroy(g));
        if (which == 1) h->launches_per_step = n;
    }
    return 0;
}

template <class K>
static int allow_smem(K kernel, int bytes) {
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return 0;
}
static int prepare_exact_kernels() {
    int rc;
    if ((rc = allow_smem(k_rmsnorm_quant<32, true>, 65536))) return rc;
    if ((rc = allow_smem(k_rmsnorm_quant<64, true>, 65536))) return rc;
    if ((rc = allow_smem(k_rmsnorm_quant<128, true>, 65536))) return rc;
#define ALLOW_GEMV(GS)                                                      \
    if ((rc = allow_smem(k_gemv<GS, EPI_STORE, true, false>, 131072))) return rc;  \
    if ((rc = allow_smem(k_gemv<GS, EPI_QKV, true, false>, 131072))) return rc;    \
    if ((rc = allow_smem(k_gemv<GS, EPI_RESID, true, false>, 131072))) return rc;  \
    if ((rc = allow_smem(k_gemv<GS, EPI_SWIGLU, true, false>, 131072))) return rc; \
    if ((rc = allow_smem(k_gemv<GS, EPI_SWIGLU, true, true>, 131072))) return rc;  \
    if ((rc = allow_smem(k_gemv<GS, EPI_STORE, false, false>, 98304))) return rc;  \
    if ((rc = allow_smem(k_gemv<GS, EPI_QKV, false, false>, 98304))) return rc;    \
    if ((rc = allow_smem(k_gemv<GS, EPI_RESID, false, false>, 98304))) return rc;  \
    if ((rc = allow_smem(k_gemv<GS, EPI_SWIGLU, false, false>, 98304))) return rc; \
    if ((rc = allow_smem(k_gemv<GS, EPI_SWIGLU, false, true>, 98304))) return rc;
    ALLOW_GEMV(32)
    ALLOW_GEMV(64)
    ALLOW_GEMV(128)
#undef ALLOW_GEMV
    return 0;
}

// ------------------------------------------------------------------------------------------
// megakernel: stream layout + launch
// ------------------------------------------------------------------------------------------
static int pick_n_kt(int K, int gs) {
    for (int n = (K + MEGA_MAX_KT - 1) / MEGA_MAX_KT; n <= 64; n++)
        if (K % (n * gs) == 0 && (K / n) % 16 == 0 && K / n <= MEGA_MAX_KT) return n;
    return 0;
}

static int build_stream(q3_handle *h, MegaGemv &g, const std::vector<const DevQT *> &src, int units, int K, bool pair) {
    const int gs = h->cfg.group_size;
    g.units = units;
    g.K = K;
    g.n_kt = pick_n_kt(K, gs);
    if (!g.n_kt) return fail(Q3_EUNSUPPORTED, "no K tiling for K=%d gs=%d", K, gs);
    g.KT = K / g.n_kt;
    g.G = g.KT / gs;
    g.tile_bytes = g.KT + ((4 * g.G + 15) & ~15);
    const size_t rows = (size_t)units * (pair ? 2 : 1);
    g.layer_stride = (long long)(rows * g.n_kt * g.tile_bytes);
    uint8_t *buf = nullptr;
    int rc;
    if ((rc = dmalloc(h, (void **)&buf, (size_t)g.layer_stride * src.size()))) return rc;
    g.base = buf;
    for (size_t l = 0; l < src.size(); l++) {
        dim3 grid(units, g.n_kt);
        GS_DISPATCH(gs, (k_build_stream<GS><<<grid, 256, 0, h->stream>>>(src[l]->q, src[l]->s, buf + l * g.layer_stride, units, K,
                                                                        g.n_kt, h->num_sms, pair ? 1 : 0)));
    }
    CK(cudaGetLastError());
    return 0;
}

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn();
// K / V cache as a 2-D f32 tensor [n_layers * seq_len rows][KV_l]; box = MEGA_KV_ROWS rows x 128 floats (one kv head), no swizzle
static int make_map_kv(CUtensorMap *map, const float *base, size_t rows, int KV_l) {
    auto enc = get_encode_fn();
    if (!enc) return fail(Q3_ECUDA, "cuTensorMapEncodeTiled unavailable");
    cuuint64_t dims[2] = {(cuuint64_t)KV_l, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)KV_l * 4};
    cuuint32_t box[2] = {(cuuint32_t)HEAD_DIM, (cuuint32_t)MEGA_KV_ROWS};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(Q3_ECUDA, "cuTensorMapEncodeTiled (KV cache) failed (%d) rows %zu KV %d", (int)r, rows, KV_l);
    return 0;
}

static int build_mega(q3_handle *h, const float *rms_att_all, const float *rms_ffn_all, const float *q_ln_all, const float *k_ln_all) {
    const q3_config &c = h->cfg;
    const int gs = c.group_size, L = c.n_layers, dim = c.dim;
    h->mega_ok = false;
    if (dim > MEGA_MAX_KT) { h->mega_why = "dim > 4096 (QKV/gate-up/lm_head phases need a single K tile)"; return 0; }
    if (!pick_n_kt(h->AH_l, gs) || !pick_n_kt(h->H_l, gs)) { h->mega_why = "no K tiling for o_proj/down"; return 0; }
    if (h->AH_l > 16384 || h->H_l > 16384 || dim > 16384) { h->mega_why = "activation vector > 16384"; return 0; }
    if (c.vocab_size % h->tp_size) { h->mega_why = "vocab not divisible by tp"; return 0; }
    // zone-reuse safety of the flagged exchanges (q3_mega.cuh): every CTA must own a qkv row and a gate/up unit
    if (h->layers[0].qkv.rows < h->num_sms || h->H_l < h->num_sms) { h->mega_why = "fewer qkv rows / FFN units than SMs"; return 0; }
    if (!get_encode_fn()) { h->mega_why = "cuTensorMapEncodeTiled unavailable"; return 0; }
    MegaArgs &a = h->margs;
    a = MegaArgs{};
    {
        int rck;
        if ((rck = make_map_kv(&a.map_k, h->kc, (size_t)L * c.seq_len, h->KV_l))) return rck;
        if ((rck = make_map_kv(&a.map_v, h->vc, (size_t)L * c.seq_len, h->KV_l))) return rck;
    }
    a.dim = dim; a.n_layers = L; a.n_heads_l = h->n_heads_l; a.n_kv_l = h->n_kv_l; a.AH_l = h->AH_l; a.KV_l = h->KV_l;
    a.H_l = h->H_l; a.seq_len = c.seq_len; a.tp_rank = h->tp_rank; a.tp_size = h->tp_size;
    a.vocab_l = c.vocab_size / h->tp_size;
    a.vocab_row0 = a.vocab_l * h->tp_rank;
    int rc;
    std::vector<const DevQT *> v;
    for (auto &W : h->layers) v.push_back(&W.qkv);
    if ((rc = build_stream(h, a.g[PH_QKV], v, h->layers[0].qkv.rows, dim, false))) return rc;
    v.clear();
    for (auto &W : h->layers) v.push_back(&W.wo);
    if ((rc = build_stream(h, a.g[PH_O], v, dim, h->AH_l, false))) return rc;
    v.clear();
    for (auto &W : h->layers) v.push_back(&W.w13);
    if ((rc = build_stream(h, a.g[PH_GU], v, h->H_l, dim, true))) return rc;
    v.clear();
    for (auto &W : h->layers) v.push_back(&W.w2);
    if ((rc = build_stream(h, a.g[PH_DN], v, dim, h->H_l, false))) return rc;
    DevQT head_slice = h->wcls; // this rank's vocab rows
    head_slice.q = h->wcls.q + (size_t)a.vocab_row0 * dim;
    head_slice.s = h->wcls.s + (size_t)a.vocab_row0 * (dim / gs);
    v.assign(1, &head_slice);
    if ((rc = build_stream(h, a.g[PH_HEAD], v, a.vocab_l, dim, false))) return rc;
    CK(cudaStreamSynchronize(h->stream));
    float *p;
    if ((rc = upload_f32(h, &p, rms_att_all, (size_t)L * dim))) return rc; a.rms_att = p;
    if ((rc = upload_f32(h, &p, rms_ffn_all, (size_t)L * dim))) return rc; a.rms_ffn = p;
    if ((rc = upload_f32(h, &p, q_ln_all, (size_t)L * HEAD_DIM))) return rc; a.q_ln = p;
    if ((rc = upload_f32(h, &p, k_ln_all, (size_t)L * HEAD_DIM))) return rc; a.k_ln = p;
    a.rms_final = h->rms_final;
    a.embed_q = h->embed.q; a.embed_s = h->embed.s; a.rope = h->rope; a.kc = h->kc; a.vc = h->vc;
    for (int i = 0; i < 2; i++) h->part_buf[i] = (unsigned long long *)(h->xchg + h->off_part[i]);
    {   // local zones, zero = "never written" (epoch 0 is not a valid epoch)
        struct { unsigned long long **p; size_t words; } zones[] = {
            {&h->zq, (size_t)h->AH_l + 2 * (size_t)h->KV_l},
            {&h->za, (size_t)h->AH_l / 4 + (size_t)h->AH_l / gs},
            {&h->zh, (size_t)h->H_l},
            {&h->zr[0], (size_t)dim},
            {&h->zr[1], (size_t)dim}};
        for (auto &z : zones) {
            if ((rc = dmalloc(h, (void **)z.p, (z.words + 2) * 8))) return rc;
            CK(cudaMemset(*z.p, 0, (z.words + 2) * 8));
        }
    }
    h->d_best = (unsigned long long *)(h->xchg + h->off_best);
    h->d_flags = (unsigned int *)(h->xchg + h->off_flags);
    if ((rc = dmalloc(h, (void **)&h->d_bar, 64))) return rc;
    CK(cudaMemset(h->d_bar, 0, 64));
    if ((rc = dmalloc(h, (void **)&h->d_status, 64))) return rc;
    CK(cudaMemset(h->d_status, 0, 64));
    int *d_status = h->d_status;
    a.x = h->x;
    a.zq = h->zq; a.za = h->za; a.zh = h->zh; a.zr[0] = h->zr[0]; a.zr[1] = h->zr[1];
    a.attn_part = h->attn_part; a.att_cnt = h->att_cnt;
    a.bar = h->d_bar; a.status = d_status; a.tokpos = h->d_tokpos; a.history = h->d_history;
    // until q3_tp_connect every "peer" slot points at this rank's own buffers
    for (int r = 0; r < MEGA_MAX_TP; r++) {
        a.part[0][r] = h->part_buf[0]; a.part[1][r] = h->part_buf[1];
        a.logits[r] = h->logits; a.best[r] = h->d_best; a.xbar[r] = (unsigned long long *)h->d_flags;
    }
    GS_DISPATCH(gs, KV_DISPATCH(h->kv_mul, (h->mega_fn = (void *)k_mega_decode<GS, KVM>)));
    if (!h->mega_fn) { h->mega_why = "no kernel for this GQA factor"; return 0; }
    const size_t slot = (size_t)MEGA_GW * (MEGA_MAX_KT + 4 * (MEGA_MAX_KT / gs));
    h->mega_smem = MEGA_NSTAGE * slot + MEGA_SCRATCH + 1024 + MEGA_MAX_KT * 4;
    CK(cudaFuncSetAttribute(h->mega_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->mega_smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, h->mega_fn, MEGA_THREADS, h->mega_smem));
    if (occ < 1) { h->mega_why = "megakernel does not fit on an SM"; return 0; }
    h->mega_ok = true;
    return 0;
}

// one cooperative launch: layers [l0, l1) (+ head).  All ranks of a TP group must issue the same sequence.
static int launch_mega(q3_handle *h, int l0, int l1, bool from_embed, bool run_head, bool feedback, bool gather) {
    MegaArgs a = h->margs;
    a.layer0 = l0; a.layer1 = l1; a.from_embed = from_embed; a.run_head = run_head; a.feedback = feedback;
    // which ranks receive this rank's vocabulary shard: every rank (each caller of q3_forward gets the full logits), or -- when a
    // logits root is configured -- the root only, on every launch (the ranks need not agree on who asked for logits)
    a.gather_logits = h->tp_size > 1 ? (h->logits_root >= 0 ? (1 << h->logits_root) : (gather ? (1 << h->tp_size) - 1 : 0)) : 0;
    a.bar_base = h->bar_base;
    a.xbar_base = h->xbar_base;
    if (h->poisoned) return fail(Q3_ECOMM, "tensor-parallel handle is unusable after a timed-out wait (ranks may have diverged): destroy and re-create every rank");
    // the only grid barrier of a launch is the one before the argmax (cross-GPU under TP); every per-layer edge is a flagged exchange
    const int nbar = run_head ? 1 : 0;
    const int nx = h->tp_size > 1 ? nbar : 0;
    a.ll_base = (unsigned)(h->ll_count % 0xFFFFFFFFull); // epochs = (count mod 2^32 - 1) + 1: never 0, wrap-around is harmless
    h->ll_count += (unsigned long long)MEGA_EDGES * (unsigned)(l1 - l0 + 1); // one epoch per step; + the head step's slot
    void *params[] = {&a};
    CK(cudaLaunchCooperativeKernel(h->mega_fn, dim3(h->num_sms), dim3(MEGA_THREADS), params, h->mega_smem, h->stream));
    h->bar_base += (unsigned long long)(nbar - nx) * h->num_sms;
    h->xbar_base += (unsigned long long)nx * h->tp_size * h->num_sms;
    return 0;
}

static int check_tok_pos(const q3_handle *h, int token, int pos);
// The end of every entry point that waits for its work: one synchronize of the handle's stream, then -- did any in-kernel wait
// time out?  The 4-byte status read is queued on the stream BEFORE the synchronize so that the check costs no extra round trip.
static int finish_call(q3_handle *h) {
    const bool mega = h->d_status && h->decode_path == 1;
    if (mega) CK(cudaMemcpyAsync(h->h_small + 16, h->d_status, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (!mega) return 0;
    const int code = h->h_small[16];
    if (code) {
        // Single GPU: all protocol state is local, reset it and the handle stays usable.  Tensor parallel: peers write into this
        // rank's flags and keep their own counters, so a rank-local reset would pair stale counters -- fail-stop instead.
        cudaMemset(h->d_status, 0, 64);
        if (h->tp_size > 1) {
            h->poisoned = true;
        } else {
            h->bar_base = 0;
            h->xbar_base = 0;
            cudaMemset(h->d_bar, 0, 64);
            cudaMemset(h->d_flags, 0, 64 * 4);
            if (h->att_cnt) cudaMemset(h->att_cnt, 0, (size_t)h->cfg.n_layers * h->n_kv_l * 4);
        }
        return fail(Q3_ECUDA, "persistent decode kernel: a wait timed out (status %d: 1 grid barrier, 2 stage ring, 3 cross-GPU barrier, 4 producer order, "
                              "6-10 flagged exchange: 6 o/down rows, 7 attention output, 8 SwiGLU outputs, 9 qkv rows, 10 TP partials; 11 prefill cross-GPU barrier)%s", code,
                    h->tp_size > 1 ? "; tensor-parallel handle poisoned" : "");
    }
    return 0;
}
extern "C" int q3_debug_profile(q3_handle *h, int token, int pos, unsigned long long *out, size_t out_words, int *n_rows_out,
                                int *n_events_out) {
    if (!h) return fail(Q3_EINVAL, "null argument");
    if (n_rows_out) *n_rows_out = 3 * h->num_sms;
    if (n_events_out) *n_events_out = MEGA_PROF_EVENTS;
    if (!out) return out_words == 0 ? Q3_OK : fail(Q3_EINVAL, "null argument"); // size query
    if (!h->mega_ok) return fail(Q3_EUNSUPPORTED, "persistent decode kernel unavailable: %s", h->mega_why.c_str());
    if (out_words < (size_t)3 * h->num_sms * MEGA_PROF_EVENTS)
        return fail(Q3_EINVAL, "profile buffer too small: %zu words, need %zu", out_words, (size_t)3 * h->num_sms * MEGA_PROF_EVENTS);
    if (int rc0 = check_tok_pos(h, token, pos)) return rc0;
    CK(cudaSetDevice(h->device));
    h->h_small[0] = token; h->h_small[1] = pos; h->h_small[2] = 0; h->h_small[3] = 0;
    CK(cudaMemcpyAsync(h->d_tokpos, h->h_small, 16, cudaMemcpyHostToDevice, h->stream));
    unsigned long long *d = nullptr;
    size_t bytes = (size_t)3 * h->num_sms * MEGA_PROF_EVENTS * 8; // consumer thread 0 rows, producer-0 rows, consumer group-1 rows
    CK(cudaMalloc((void **)&d, bytes));
    CK(cudaMemsetAsync(d, 0, bytes, h->stream));
    h->margs.prof = d;
    int rc = launch_mega(h, 0, h->cfg.n_layers, true, true, false, false);
    h->margs.prof = nullptr;
    if (!rc) { // the stamps are copied out even when a wait timed out: they show where
        cudaError_t e = cudaMemcpyAsync(out, d, bytes, cudaMemcpyDeviceToHost, h->stream);
        rc = e == cudaSuccess ? finish_call(h) : fail(Q3_ECUDA, "profile copy failed: %s", cudaGetErrorString(e));
    }
    cudaFree(d);
    return rc;
}
extern "C" int q3_num_sms(const q3_handle *h) { return h ? h->num_sms : 0; }
// test hook: move the flagged-exchange epoch counter (e.g. next to the 2^32 - 1 wrap); all TP ranks must use the same value
extern "C" int q3_debug_set_epoch(q3_handle *h, unsigned long long exchanges_issued) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    h->ll_count = exchanges_issued;
    return Q3_OK;
}

static inline bool use_mega(const q3_handle *h) { return h->decode_path == 1 && h->mega_ok && !h->exact; }
static int tp_ready(const q3_handle *h) {
    if (h->tp_size > 1 && !h->tp_connected) return fail(Q3_ECOMM, "tensor-parallel handle used before q3_tp_connect");
    if (h->tp_size > 1 && !use_mega(h)) return fail(Q3_EUNSUPPORTED, "under tensor parallelism only the persistent fast path is available");
    return 0;
}

// what a caller needs from one decode step
enum StepOut {
    STEP_LOGITS,   // the logits
    STEP_ARGMAX,   // + their argmax in d_tokpos[2]
    STEP_FEEDBACK, // + the argmax fed back as the next token / position and appended to the history
};
// One decode step of the token / position in d_tokpos on the current path: the persistent kernel, or the CUDA graph of the
// exact mask.  gather: see launch_mega.
static int launch_decode_step(q3_handle *h, StepOut out, bool gather = false) {
    if (use_mega(h)) return launch_mega(h, 0, h->cfg.n_layers, true, true, out == STEP_FEEDBACK, gather);
    CK(cudaGraphLaunch(out == STEP_FEEDBACK ? h->g_greedy[h->exact] : h->g_fwd[h->exact], h->stream));
    if (out == STEP_ARGMAX) launch_argmax(h, false, h->stream);
    return 0;
}
// final norm + lm_head on h->x alone
static int launch_head_only(q3_handle *h, bool gather) {
    if (use_mega(h)) return launch_mega(h, 0, 0, false, true, false, gather);
    launch_head(h, h->stream);
    return 0;
}

// ------------------------------------------------------------------------------------------
// batched prefill: tcgen05 int8 GEMM (q3_prefill.cuh) + batched norm / rope / attention
// ------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
    }
    return fn;
}
// 2-D int8 matrix [rows][K] (row pitch K bytes), box = 128 rows x 128 bytes, 128B swizzle
static int make_map_i8(CUtensorMap *map, const void *base, int rows, int K) {
    auto enc = get_encode_fn();
    if (!enc) return fail(Q3_ECUDA, "cuTensorMapEncodeTiled unavailable");
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)K};
    cuuint32_t box[2] = {(cuuint32_t)PF_BK, (cuuint32_t)PF_BM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(Q3_ECUDA, "cuTensorMapEncodeTiled failed (%d) rows %d K %d", (int)r, rows, K);
    return 0;
}

// group-major scale matrix [groups][cols] f32 (row pitch cols * 4 bytes), box = 2 groups x 128 columns: the scale rows of one
// accumulator pair arrive with ONE tensor copy
static int make_map_scales(CUtensorMap *map, const float *base, int groups, int cols) {
    auto enc = get_encode_fn();
    if (!enc) return fail(Q3_ECUDA, "cuTensorMapEncodeTiled unavailable");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)groups};
    cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
    cuuint32_t box[2] = {128, 2};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(Q3_ECUDA, "cuTensorMapEncodeTiled (scales) failed (%d) groups %d cols %d", (int)r, groups, cols);
    return 0;
}

template <int GS, int EPI, bool EXACT>
static int launch_gemm_q8_t(const CUtensorMap &mx, const CUtensorMap &mw, const PrefillGemmArgs &a, cudaStream_t s) {
    static bool attr = false;
    if (!attr) {
        CK(cudaFuncSetAttribute(k_gemm_q8<GS, EPI, EXACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
        attr = true;
    }
    static int num_sms = 0;
    if (!num_sms) {
        int dev = 0;
        CK(cudaGetDevice(&dev));
        CK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    }
    CUtensorMap mxs, mws;
    int rc;
    if ((rc = make_map_scales(&mxs, a.xsT, a.K / GS, a.Tpad)) || (rc = make_map_scales(&mws, a.wsT, a.K / GS, a.N))) return rc;
    const int tiles = (a.N / PF_BN) * (a.Tpad / PF_BM); // persistent: one CTA per SM walks the tiles
    k_gemm_q8<GS, EPI, EXACT><<<tiles < num_sms ? tiles : num_sms, PF_THREADS, PF_SMEM, s>>>(mx, mw, mxs, mws, a);
    return 0;
}
// mode 0: the fast drain (what q3_prefill runs); 1: the exact drain, reference-order f32 fold (bit-identical to matmul), built
// for the plain store epilogue only -- the operator and timing entry points are its only callers.  The int32 group dots are
// the same in both modes.
template <int EPI>
static int launch_gemm_q8(int gs, const CUtensorMap &mx, const CUtensorMap &mw, const PrefillGemmArgs &a, cudaStream_t s, int mode = 0) {
    int rc = 0;
    if (mode == 0) {
        GS_DISPATCH(gs, (rc = launch_gemm_q8_t<GS, EPI, false>(mx, mw, a, s)));
    } else if (mode == 1 && EPI == PF_EPI_STORE) {
        GS_DISPATCH(gs, (rc = launch_gemm_q8_t<GS, PF_EPI_STORE, true>(mx, mw, a, s)));
    } else {
        return fail(Q3_EINVAL, "prefill GEMM mode %d: 0 = fast drain, 1 = exact drain (plain store epilogue only)", mode);
    }
    return rc;
}

// group-major scales + TMA map for one weight tensor
static int prefill_prepare_tensor(q3_handle *h, DevQT &t) {
    if (t.has_map) return 0;
    const int gs = h->cfg.group_size, ng = t.K / gs;
    int rc;
    if ((rc = dmalloc(h, (void **)&t.sT, (size_t)ng * t.rows * 4))) return rc;
    dim3 grid((ng + 31) / 32, (t.rows + 31) / 32);
    k_transpose_f32<<<grid, dim3(32, 8), 0, h->stream>>>(t.s, t.sT, t.rows, ng);
    CK(cudaGetLastError());
    if ((rc = make_map_i8(&t.map, t.q, t.rows, t.K))) return rc;
    t.has_map = true;
    return 0;
}

// k_pf_attention_h needs more than the default 48 KB of dynamic shared memory
static int allow_pf_attention(int kv_mul) {
    int rc = 0;
    KV_DISPATCH(kv_mul, (rc = allow_smem(k_pf_attention_h<KVM>, PFH_SMEM)));
    return rc;
}

// causal attention of T query rows (positions pos0 .. pos0+T-1) over K / V cache rows 0 .. pos0+T-1 on the tensor cores, FP16
// hi / lo split: the K / V rows are split once into kvh ([4][plane] halves), then streamed
static void launch_pf_attention(const float *q, const float *kc, const float *vc, __half *kvh, size_t plane, float *out, int T, int pos0,
                                int n_kv, int kv_mul, int num_sms, cudaStream_t s) {
    const int AH = n_kv * kv_mul * HEAD_DIM, KV = n_kv * HEAD_DIM;
    k_pf_split_kv<<<num_sms * 4, 256, 0, s>>>(kc, vc, kvh, ((size_t)pos0 + T) * KV / 4, plane);
    const int bq = PFH_R / kv_mul;
    dim3 ag(n_kv, (T + bq - 1) / bq);
    KV_DISPATCH(kv_mul, (k_pf_attention_h<KVM><<<ag, 128, PFH_SMEM, s>>>(q, kvh, plane, out, T, pos0, AH, KV)));
}

// RMSNorm + quantise of rows [0, T) of x (pitch dim) into pf_xq / pf_xsT (group-major, pitch Tpad); embed: the rows are first
// gathered from the embedding table at pf_tokens
static void launch_pf_norm_quant(const q3_handle *h, float *x, const float *w, int T, int Tpad, bool embed) {
    const int dim = h->cfg.dim;
    const int8_t *eq = embed ? h->embed.q : nullptr;
    if (dim <= 4096) {
        GS_DISPATCH(h->cfg.group_size, (k_pf_norm_quant<GS, 4><<<T, 256, 0, h->stream>>>(x, w, h->pf_xq, h->pf_xsT, dim, Tpad, eq, h->embed.s, h->pf_tokens, 0)));
    } else {
        GS_DISPATCH(h->cfg.group_size, (k_pf_norm_quant<GS><<<T, 256, 0, h->stream>>>(x, w, h->pf_xq, h->pf_xsT, dim, Tpad, eq, h->embed.s, h->pf_tokens, 0)));
    }
}

static int prefill_init(q3_handle *h) {
    const q3_config &c = h->cfg;
    h->pf_ok = false;
    if (c.dim % 128 || h->AH_l % 128 || h->H_l % 128 || h->layers[0].qkv.rows % 128 || (2 * h->H_l) % 128) {
        h->pf_why = "matrix dimensions must be multiples of 128";
        return 0;
    }
    if ((c.dim / c.group_size) % 2 || (h->AH_l / c.group_size) % 2 || (h->H_l / c.group_size) % 2) {
        h->pf_why = "the tensor-core GEMM hands accumulators over in pairs: rows need an even number of quantisation groups";
        return 0;
    }
    if (!get_encode_fn()) { h->pf_why = "cuTensorMapEncodeTiled unavailable"; return 0; }
    int rc;
    if ((rc = allow_pf_attention(h->kv_mul))) return rc;
    for (auto &W : h->layers) {
        if ((rc = prefill_prepare_tensor(h, W.qkv))) return rc;
        if ((rc = prefill_prepare_tensor(h, W.wo))) return rc;
        if ((rc = prefill_prepare_tensor(h, W.w13))) return rc;
        if ((rc = prefill_prepare_tensor(h, W.w2))) return rc;
    }
    CK(cudaStreamSynchronize(h->stream));
    h->pf_ok = true;
    return 0;
}

static void prefill_release(q3_handle *h) {
    if (h->pf_kvh) cudaFree(h->pf_kvh);
    h->pf_kvh = nullptr;
    h->pf_kvh_rows = 0;
    void **ps[] = {(void **)&h->pf_x, (void **)&h->pf_q, (void **)&h->pf_att, (void **)&h->pf_hb, (void **)&h->pf_xsT, (void **)&h->pf_hsT,
                   (void **)&h->pf_xq, (void **)&h->pf_hq, (void **)&h->pf_tokens};
    for (void **p : ps) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    h->pf_cap = 0;
}
static int prefill_reserve(q3_handle *h, int T) {
    const int Tpad = (T + 127) / 128 * 128;
    if (Tpad <= h->pf_cap) return 0;
    const q3_config &c = h->cfg;
    const int gs = c.group_size, dim = c.dim, AH = h->AH_l, H = h->H_l;
    const int maxd = AH > dim ? AH : dim;
    prefill_release(h);
    struct { void **p; size_t bytes; } want[] = {
        {(void **)&h->pf_x, (size_t)Tpad * dim * 4},          {(void **)&h->pf_q, (size_t)Tpad * AH * 4},
        {(void **)&h->pf_att, (size_t)Tpad * AH * 4},         {(void **)&h->pf_hb, (size_t)Tpad * H * 4},
        {(void **)&h->pf_xsT, (size_t)(maxd / gs) * Tpad * 4}, {(void **)&h->pf_hsT, (size_t)(H / gs) * Tpad * 4},
        {(void **)&h->pf_xq, (size_t)Tpad * maxd},            {(void **)&h->pf_hq, (size_t)Tpad * H},
        {(void **)&h->pf_tokens, (size_t)Tpad * 4}};
    for (auto &w : want) {
        cudaError_t e = cudaMalloc(w.p, w.bytes);
        if (e != cudaSuccess) { // leave no dangling pointer behind: a later prefill / destroy must not free twice
            *w.p = nullptr;
            prefill_release(h);
            cudaGetLastError();
            return fail(Q3_ECUDA, "prefill buffers for %d tokens: %s", T, cudaGetErrorString(e));
        }
    }
    CK(cudaMemset(h->pf_xq, 0, (size_t)Tpad * maxd));
    CK(cudaMemset(h->pf_hq, 0, (size_t)Tpad * H));
    CK(cudaMemset(h->pf_xsT, 0, (size_t)(maxd / gs) * Tpad * 4));
    CK(cudaMemset(h->pf_hsT, 0, (size_t)(H / gs) * Tpad * 4));
    h->pf_cap = Tpad;
    return 0;
}

// Row-parallel GEMM under tensor parallelism (o_proj: which = 0, down_proj: which = 1): partial block -> exchange buffer, cross-GPU
// barrier, rank-ordered sum of the tp partials over NVLink folded into the residual stream (q3_prefill.cuh).  All ranks issue the
// same sequence, so the barrier count is the same everywhere.
static int prefill_tp_rowparallel(q3_handle *h, int which, const CUtensorMap &mx, const CUtensorMap &mw, PrefillGemmArgs g, int T) {
    int rc;
    g.out = const_cast<float *>(h->pf_peers[which].part[h->tp_rank]);
    if ((rc = launch_gemm_q8<PF_EPI_STORE>(h->cfg.group_size, mx, mw, g, h->stream))) return rc;
    h->pf_xbar_count++;
    k_pf_xbarrier<<<1, 32, 0, h->stream>>>(h->pf_peers[which], h->tp_size, h->tp_rank, h->pf_xbar_count * (unsigned long long)h->tp_size, h->d_status);
    const size_t n4 = (size_t)T * h->cfg.dim / 4;
    // tp > 2: reduce-scatter, barrier, all-gather -- 2 (tp-1)/tp blocks over NVLink instead of tp-1.  At tp 2 both move one block,
    // and the one-pass all-reduce saves the second barrier.
    if (h->tp_size > 2) {
        k_pf_reduce_scatter<<<h->num_sms * 2, 256, 0, h->stream>>>(h->pf_peers[which], g.out, h->tp_size, h->tp_rank, n4);
        h->pf_xbar_count++;
        k_pf_xbarrier<<<1, 32, 0, h->stream>>>(h->pf_peers[which], h->tp_size, h->tp_rank, h->pf_xbar_count * (unsigned long long)h->tp_size, h->d_status);
        k_pf_allgather_resid<<<dim3(h->num_sms / 2, h->tp_size), 256, 0, h->stream>>>(h->pf_x, h->pf_peers[which], h->tp_size, n4);
    } else {
        k_pf_allreduce_resid<<<h->num_sms * 4, 256, 0, h->stream>>>(h->pf_x, h->pf_peers[which], h->tp_size, n4);
    }
    CK(cudaGetLastError());
    return 0;
}

static int prefill_run(q3_handle *h, const int *tokens_host, int T, int pos0);
static int score_rows(q3_handle *h, int T, int out0);
// prompts longer than the tensor-parallel partial blocks go through in chunks (causal attention reads the earlier chunks' cache rows).
// score: q3_score's head stage on each chunk's rows of pf_x, before the next chunk overwrites them.
static int prefill_chunks(q3_handle *h, const int *tokens_host, int n, int pos0, bool score = false) {
    const int cap = h->tp_size > 1 ? h->pf_tp_cap : n;
    for (int off = 0; off < n; off += cap) {
        const int T = n - off < cap ? n - off : cap;
        int rc = prefill_run(h, tokens_host + off, T, pos0 + off);
        if (!rc && score) rc = score_rows(h, T, off);
        if (rc) return rc;
    }
    return 0;
}

// the whole batched forward for tokens at positions pos0..pos0+T-1; leaves x of the last token in h->x
static int prefill_run(q3_handle *h, const int *tokens_host, int T, int pos0) {
    const q3_config &c = h->cfg;
    const int gs = c.group_size, dim = c.dim, AH = h->AH_l, KV = h->KV_l, H = h->H_l;
    int rc;
    if ((rc = prefill_reserve(h, T))) return rc;
    if ((size_t)pos0 + T > h->pf_kvh_rows) { // hi / lo copy of one layer's K / V rows (grow-only)
        if (h->pf_kvh) cudaFree(h->pf_kvh);
        h->pf_kvh = nullptr;
        h->pf_kvh_rows = 0;
        const size_t rows = ((size_t)pos0 + T + 127) / 128 * 128;
        cudaError_t e = cudaMalloc((void **)&h->pf_kvh, 4 * rows * KV * sizeof(__half));
        if (e != cudaSuccess) {
            h->pf_kvh = nullptr;
            cudaGetLastError();
            return fail(Q3_ECUDA, "prefill K/V split buffer for %zu rows: %s", rows, cudaGetErrorString(e));
        }
        h->pf_kvh_rows = rows;
    }
    const int Tpad = (T + 127) / 128 * 128;
    cudaStream_t s = h->stream;
    CK(cudaMemcpyAsync(h->pf_tokens, tokens_host, (size_t)T * 4, cudaMemcpyHostToDevice, s));
    CUtensorMap mx_dim, mx_ah, mx_h;
    if ((rc = make_map_i8(&mx_dim, h->pf_xq, Tpad, dim))) return rc;
    if ((rc = make_map_i8(&mx_ah, h->pf_xq, Tpad, AH))) return rc;
    if ((rc = make_map_i8(&mx_h, h->pf_hq, Tpad, H))) return rc;
    for (int l = 0; l < c.n_layers; l++) {
        LayerDev &W = h->layers[l];
        float *kc_l = h->kc + (size_t)l * c.seq_len * KV;
        float *vc_l = h->vc + (size_t)l * c.seq_len * KV;
        // attn_norm + quantize (qwen3.rs:134-136), embedding on layer 0
        launch_pf_norm_quant(h, h->pf_x, W.rms_att, T, Tpad, l == 0);
        PrefillGemmArgs g{};
        g.T = T; g.Tpad = Tpad; g.K = dim; g.N = W.qkv.rows; g.wsT = W.qkv.sT; g.xsT = h->pf_xsT;
        g.q = h->pf_q; g.kc = kc_l; g.vc = vc_l; g.AH = AH; g.KV = KV; g.pos0 = pos0;
        if ((rc = launch_gemm_q8<PF_EPI_QKV>(gs, mx_dim, W.qkv.map, g, s))) return rc;
        dim3 rg((h->n_heads_l + h->n_kv_l + 3) / 4, T);
        k_pf_qknorm_rope<<<rg, 128, 0, s>>>(h->pf_q, kc_l, W.q_ln, W.k_ln, h->rope, pos0, h->n_heads_l, h->n_kv_l, AH, KV);
        launch_pf_attention(h->pf_q, kc_l, vc_l, h->pf_kvh, h->pf_kvh_rows * KV, h->pf_att, T, pos0, h->n_kv_l, h->kv_mul, h->num_sms, s);
        GS_DISPATCH(gs, (k_pf_quantize<GS><<<T, 256, 0, s>>>(h->pf_att, h->pf_xq, h->pf_xsT, AH, Tpad)));
        PrefillGemmArgs o{};
        o.T = T; o.Tpad = Tpad; o.K = AH; o.N = dim; o.wsT = W.wo.sT; o.xsT = h->pf_xsT; o.out = h->pf_x; o.ld_out = dim;
        if (h->tp_size == 1) {
            if ((rc = launch_gemm_q8<PF_EPI_RESID>(gs, mx_ah, W.wo.map, o, s))) return rc;
        } else if ((rc = prefill_tp_rowparallel(h, 0, mx_ah, W.wo.map, o, T))) return rc;
        launch_pf_norm_quant(h, h->pf_x, W.rms_ffn, T, Tpad, false);
        PrefillGemmArgs gu{};
        gu.T = T; gu.Tpad = Tpad; gu.K = dim; gu.N = W.w13.rows; gu.wsT = W.w13.sT; gu.xsT = h->pf_xsT; gu.out = h->pf_hb; gu.ld_out = H;
        if ((rc = launch_gemm_q8<PF_EPI_SWIGLU>(gs, mx_dim, W.w13.map, gu, s))) return rc;
        GS_DISPATCH(gs, (k_pf_quantize<GS><<<T, 256, 0, s>>>(h->pf_hb, h->pf_hq, h->pf_hsT, H, Tpad)));
        PrefillGemmArgs dn{};
        dn.T = T; dn.Tpad = Tpad; dn.K = H; dn.N = dim; dn.wsT = W.w2.sT; dn.xsT = h->pf_hsT; dn.out = h->pf_x; dn.ld_out = dim;
        if (h->tp_size == 1) {
            if ((rc = launch_gemm_q8<PF_EPI_RESID>(gs, mx_h, W.w2.map, dn, s))) return rc;
        } else if ((rc = prefill_tp_rowparallel(h, 1, mx_h, W.w2.map, dn, T))) return rc;
    }
    CK(cudaMemcpyAsync(h->x, h->pf_x + (size_t)(T - 1) * dim, (size_t)dim * 4, cudaMemcpyDeviceToDevice, s));
    CK(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------
// q3_score: final norm + lm_head + log-softmax / argmax on every row of the batched prefill
// ------------------------------------------------------------------------------------------
// lm_head rows per GEMM: a [T][vocab] f32 block would be 1.24 GB at T 2048 (151936 entries), so the head runs in row chunks
constexpr int SCORE_ROWS = 512;

// the per-position buffers [seq_len]; with lm_head: also the lm_head's group-major scales / TMA map and room for `rows` logits
// rows.  Grow-only; nothing is allocated before the first q3_score.
static int score_reserve(q3_handle *h, bool lm_head, int rows) {
    const q3_config &c = h->cfg;
    int rc;
    if (!h->sc_targets) { // one allocation: a failure leaves all three unset
        int *p = nullptr;
        if ((rc = dmalloc(h, (void **)&p, (size_t)c.seq_len * 12))) return rc;
        h->sc_targets = p;
        h->sc_argmax = p + c.seq_len;
        h->sc_lp = (float *)(p + 2 * (size_t)c.seq_len);
    }
    if (!lm_head) return 0;
    if ((rc = prefill_prepare_tensor(h, h->wcls))) return rc; // tied: sets sT / map on the copy in wcls only, freed once with allocs
    rows = (rows + 127) / 128 * 128;
    if (rows > SCORE_ROWS) rows = SCORE_ROWS;
    if (rows <= h->sc_cap) return 0;
    if (h->sc_logits) cudaFree(h->sc_logits);
    h->sc_logits = nullptr;
    h->sc_cap = 0;
    cudaError_t e = cudaMalloc((void **)&h->sc_logits, (size_t)rows * c.vocab_size * 4);
    if (e != cudaSuccess) {
        h->sc_logits = nullptr;
        cudaGetLastError();
        return fail(Q3_ECUDA, "score logits buffer for %d rows: %s", rows, cudaGetErrorString(e));
    }
    h->sc_cap = rows;
    return 0;
}

// the [seq_len][k] results of q3_score_topk, sized for the largest k asked for so far (one allocation: ids, then lps)
static int topk_reserve(q3_handle *h, int k) {
    if (k <= h->tk_cap) return 0;
    if (h->tk_ids) cudaFree(h->tk_ids);
    h->tk_ids = nullptr;
    h->tk_lps = nullptr;
    h->tk_cap = 0;
    const size_t n = (size_t)h->cfg.seq_len * k;
    cudaError_t e = cudaMalloc((void **)&h->tk_ids, n * 8);
    if (e != cudaSuccess) {
        h->tk_ids = nullptr;
        cudaGetLastError();
        return fail(Q3_ECUDA, "top-k buffers for k %d: %s", k, cudaGetErrorString(e));
    }
    h->tk_lps = (float *)(h->tk_ids + n);
    h->tk_cap = k;
    return 0;
}

static void launch_logprobs(q3_handle *h, const float *logits, int rows, int out0) {
    const int V = h->cfg.vocab_size, k = h->tk_k;
    float *lp = h->sc_want_lp ? h->sc_lp + out0 : nullptr;
    if (k)
        k_topk_logprobs<<<rows, LP_THREADS, 0, h->stream>>>(logits, V, (size_t)V, k, h->tk_ids + (size_t)out0 * k,
                                                            h->tk_lps + (size_t)out0 * k, h->sc_targets + out0, lp, h->sc_argmax + out0);
    else
        k_logprobs<<<rows, LP_THREADS, 0, h->stream>>>(logits, V, (size_t)V, h->sc_targets + out0, lp, h->sc_argmax + out0);
}

// rows [0, T) of pf_x (positions out0 .. out0 + T - 1 of the q3_score call): final RMSNorm + quantise into rows [0, Tc) of
// pf_xq / pf_xsT (pf_x is read only), the lm_head on the fast-drain tensor-core GEMM, then k_logprobs -- SCORE_ROWS rows at a time
static int score_rows(q3_handle *h, int T, int out0) {
    const q3_config &c = h->cfg;
    const int gs = c.group_size, dim = c.dim;
    cudaStream_t s = h->stream;
    int rc;
    for (int r0 = 0; r0 < T; r0 += SCORE_ROWS) {
        const int Tc = T - r0 < SCORE_ROWS ? T - r0 : SCORE_ROWS, Tcpad = (Tc + 127) / 128 * 128;
        float *x = h->pf_x + (size_t)r0 * dim;
        launch_pf_norm_quant(h, x, h->rms_final, Tc, Tcpad, false);
        CUtensorMap mx;
        if ((rc = make_map_i8(&mx, h->pf_xq, Tcpad, dim))) return rc;
        PrefillGemmArgs g{};
        g.T = Tc; g.Tpad = Tcpad; g.K = dim; g.N = c.vocab_size; g.wsT = h->wcls.sT; g.xsT = h->pf_xsT; g.out = h->sc_logits; g.ld_out = c.vocab_size;
        if ((rc = launch_gemm_q8<PF_EPI_STORE>(gs, mx, h->wcls.map, g, s))) return rc;
        launch_logprobs(h, h->sc_logits, Tc, out0 + r0);
    }
    CK(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------
// construction
// ------------------------------------------------------------------------------------------
static int create_impl(const char *path, int ctx_len, int device, int tp_rank, int tp_size, q3_handle **out) {
    if (!path || !out) return fail(Q3_EINVAL, "null argument");
    if (tp_size < 1 || tp_rank < 0 || tp_rank >= tp_size) return fail(Q3_EINVAL, "bad tp rank/size %d/%d", tp_rank, tp_size);
    *out = nullptr;
    Ckpt ck;
    int rc = open_ckpt(path, ctx_len, ck);
    if (rc) return rc;
    const q3_config &c = ck.cfg;
    const int gs = c.group_size;
    if (c.head_dim != HEAD_DIM) return fail(Q3_EUNSUPPORTED, "head_dim %d unsupported (kernels are built for 128)", c.head_dim);
    if (gs != 32 && gs != 64 && gs != 128) return fail(Q3_EUNSUPPORTED, "group_size %d unsupported (32/64/128)", gs);
    if (c.n_heads % c.n_kv_heads) return fail(Q3_EUNSUPPORTED, "n_heads %% n_kv_heads != 0");
    int kv_mul = c.n_heads / c.n_kv_heads;
    if (kv_mul != 1 && kv_mul != 2 && kv_mul != 4 && kv_mul != 8) return fail(Q3_EUNSUPPORTED, "GQA factor %d unsupported", kv_mul);
    if (c.dim % 128 || c.hidden_dim % 128) return fail(Q3_EUNSUPPORTED, "dim/hidden_dim must be multiples of 128");
    if (c.dim > 16384 || c.hidden_dim > 65536) return fail(Q3_EUNSUPPORTED, "dim/hidden_dim too large");
    if (c.n_kv_heads % tp_size || (c.hidden_dim / tp_size) % gs || c.hidden_dim % tp_size)
        return fail(Q3_EUNSUPPORTED, "tp_size %d does not divide kv heads / hidden groups", tp_size);
    if (c.vocab_size % 2) return fail(Q3_EUNSUPPORTED, "odd vocab_size");

    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(Q3_EINVAL, "device %d out of range (%d visible)", device, ndev);
    CK(cudaSetDevice(device));
    q3_handle *h = new q3_handle();
    h->cfg = c;
    h->device = device;
    h->tp_rank = tp_rank;
    h->tp_size = tp_size;
    h->kv_mul = kv_mul;
    h->n_heads_l = c.n_heads / tp_size;
    h->n_kv_l = c.n_kv_heads / tp_size;
    h->AH_l = h->n_heads_l * HEAD_DIM;
    h->KV_l = h->n_kv_l * HEAD_DIM;
    h->H_l = c.hidden_dim / tp_size;
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    h->num_sms = prop.multiProcessorCount;

    auto guard_fail = [&](int code) {
        q3_destroy(h);
        return code;
    };
#define TRY(x)                         \
    do {                               \
        int rc_ = (x);                 \
        if (rc_) return guard_fail(rc_); \
    } while (0)
#define CKH(call)                                                                                         \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return guard_fail(fail(Q3_ECUDA, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e_), __FILE__, \
                                   __LINE__, cudaGetErrorString(e_)));                                    \
    } while (0)

    CKH(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    const int L = c.n_layers, dim = c.dim, H = c.hidden_dim;
    const int AH = c.n_heads * HEAD_DIM;
    Stager st;
    h->layers.resize(L);
    const int r = tp_rank;
    for (int l = 0; l < L; l++) {
        LayerDev &W = h->layers[l];
        // column-parallel: this rank's q heads / kv heads (rows of the [out,in] matrices)
        TRY(upload_rows(h, st, W.qkv,
                        {{ck.wq[l], r * h->AH_l, h->AH_l, dim}, {ck.wk[l], r * h->KV_l, h->KV_l, dim}, {ck.wv[l], r * h->KV_l, h->KV_l, dim}},
                        dim, 0, gs));
        // row-parallel: all rows, this rank's input columns
        TRY(upload_rows(h, st, W.wo, {{ck.wo[l], 0, dim, AH}}, h->AH_l, r * h->AH_l, gs));
        TRY(upload_rows(h, st, W.w13, {{ck.w1[l], r * h->H_l, h->H_l, dim}, {ck.w3[l], r * h->H_l, h->H_l, dim}}, dim, 0, gs, true));
        TRY(upload_rows(h, st, W.w2, {{ck.w2[l], 0, dim, H}}, h->H_l, r * h->H_l, gs));
        TRY(upload_f32(h, &W.rms_att, ck.rms_att + (size_t)l * dim, dim));
        TRY(upload_f32(h, &W.rms_ffn, ck.rms_ffn + (size_t)l * dim, dim));
        TRY(upload_f32(h, &W.q_ln, ck.q_ln + (size_t)l * HEAD_DIM, HEAD_DIM));
        TRY(upload_f32(h, &W.k_ln, ck.k_ln + (size_t)l * HEAD_DIM, HEAD_DIM));
    }
    // embedding table stays int8 and is dequantised per row on the fly (bit-identical to the
    // reference's load-time dequantize, tensor.rs:72-80: a single multiply per element)
    TRY(upload_rows(h, st, h->embed, {{ck.embed, 0, c.vocab_size, dim}}, dim, 0, gs));
    if (c.shared_classifier) h->wcls = h->embed;
    else TRY(upload_rows(h, st, h->wcls, {{ck.wcls, 0, c.vocab_size, dim}}, dim, 0, gs));
    TRY(upload_f32(h, &h->rms_final, ck.rms_final, dim));

    // RoPE table on the host with glibc powf/cosf/sinf (layers.rs:161-171), one row per position
    {
        size_t n = (size_t)c.seq_len * HEAD_DIM;
        std::vector<float> tab(n);
        const int half = HEAD_DIM / 2;
        std::vector<float> freq(half);
        for (int i = 0; i < half; i++) freq[i] = powf(1e6f, -((float)i) / (float)half);
        for (int p = 0; p < c.seq_len; p++)
            for (int i = 0; i < half; i++) {
                float ang = (float)p * freq[i];
                tab[(size_t)p * HEAD_DIM + 2 * i] = cosf(ang);
                tab[(size_t)p * HEAD_DIM + 2 * i + 1] = sinf(ang);
            }
        TRY(upload_f32(h, &h->rope, tab.data(), n));
    }
    // buffers (qwen3.rs:420-444)
    const int maxd = (h->AH_l > dim ? h->AH_l : dim);
    TRY(dmalloc(h, (void **)&h->x, (size_t)dim * 4));
    TRY(dmalloc(h, (void **)&h->xb, (size_t)maxd * 4));
    TRY(dmalloc(h, (void **)&h->q, (size_t)h->AH_l * 4));
    TRY(dmalloc(h, (void **)&h->hb, (size_t)h->H_l * 4));
    {   // exchange buffer (see q3_handle::xchg); logits live inside it
        auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
        size_t o = 0;
        h->off_part[0] = o; o = al(o + (size_t)tp_size * dim * 8); // (value, epoch) words
        h->off_part[1] = o; o = al(o + (size_t)tp_size * dim * 8);
        h->off_best = o; o = al(o + (size_t)tp_size * h->num_sms * 8);
        h->off_flags = o; o = al(o + 64 * 4);
        h->off_logits = o; o = al(o + (size_t)c.vocab_size * 4);
        if (tp_size > 1) { // batched prefill: partial blocks of the row-parallel GEMMs (chunks of up to 2048 tokens)
            h->pf_tp_cap = c.seq_len < 2048 ? (c.seq_len + 127) / 128 * 128 : 2048;
            h->off_pf_ctr = o; o = al(o + 64);
            for (int i = 0; i < 2; i++) { h->off_pf_part[i] = o; o = al(o + (size_t)h->pf_tp_cap * dim * 4); }
        }
        h->xchg_bytes = o;
        TRY(dmalloc(h, (void **)&h->xchg, o));
        CKH(cudaMemset(h->xchg, 0, o));
        h->logits = (float *)(h->xchg + h->off_logits);
    }
    TRY(dmalloc(h, (void **)&h->xq, (size_t)maxd));
    TRY(dmalloc(h, (void **)&h->xs, (size_t)(maxd / gs + 1) * 4));
    TRY(dmalloc(h, (void **)&h->hq, (size_t)h->H_l));
    TRY(dmalloc(h, (void **)&h->hs, (size_t)(h->H_l / gs + 1) * 4));
    TRY(dmalloc(h, (void **)&h->attn_part, (size_t)h->n_heads_l * ATTN_MAX_SPLITS * ATTN_PART_STRIDE * 4));
    TRY(dmalloc(h, (void **)&h->att_cnt, (size_t)h->cfg.n_layers * h->n_kv_l * 4));
    CKH(cudaMemset(h->att_cnt, 0, (size_t)h->cfg.n_layers * h->n_kv_l * 4));
    TRY(dmalloc(h, (void **)&h->att, (size_t)h->n_heads_l * c.seq_len * 4));
    TRY(prepare_exact_kernels());
    size_t kvn = (size_t)L * c.seq_len * h->KV_l;
    TRY(dmalloc(h, (void **)&h->kc, kvn * 4));
    TRY(dmalloc(h, (void **)&h->vc, kvn * 4));
    CKH(cudaMemset(h->kc, 0, kvn * 4)); // vec![0.0; ..] (qwen3.rs:439-440)
    CKH(cudaMemset(h->vc, 0, kvn * 4));
    h->history_cap = c.seq_len + 8;
    TRY(dmalloc(h, (void **)&h->d_tokpos, 16 * 4));
    TRY(dmalloc(h, (void **)&h->d_history, (size_t)h->history_cap * 4));
    CKH(cudaMemset(h->d_tokpos, 0, 16 * 4));
    CKH(cudaMemset(h->x, 0, (size_t)dim * 4));
    CKH(cudaMallocHost((void **)&h->h_logits, (size_t)c.vocab_size * 4));
    CKH(cudaMallocHost((void **)&h->h_small, 64 * 4));
    CKH(cudaDeviceSynchronize());
    TRY(build_graphs(h));
    h->graph_launches_per_step = h->launches_per_step;
    TRY(build_mega(h, ck.rms_att, ck.rms_ffn, ck.q_ln, ck.k_ln));
    if (h->mega_ok) {
        h->decode_path = 1;
        h->launches_per_step = 1;
    }
    TRY(prefill_init(h));
    CKH(cudaDeviceSynchronize());
    *out = h;
    return Q3_OK;
}

extern "C" int q3_create(const char *path, int ctx_len, int device, q3_handle **out) {
    return create_impl(path, ctx_len, device, 0, 1, out);
}
extern "C" int q3_create_tp(const char *path, int ctx_len, int device, int tp_rank, int tp_size, q3_handle **out) {
    if (tp_size > MEGA_MAX_TP) return fail(Q3_EUNSUPPORTED, "tp_size %d > %d", tp_size, MEGA_MAX_TP);
    int rc = create_impl(path, ctx_len, device, tp_rank, tp_size, out);
    if (rc) return rc;
    if (tp_size > 1 && !(*out)->mega_ok) {
        std::string why = (*out)->mega_why;
        q3_destroy(*out);
        *out = nullptr;
        return fail(Q3_EUNSUPPORTED, "tensor parallelism needs the persistent decode kernel, unavailable here: %s", why.c_str());
    }
    return Q3_OK;
}

// blob exchanged between ranks (all-gathered by the host): who I am + how to map my exchange buffer
struct TpBlob {
    uint32_t magic, rank, tp_size, device;
    uint64_t pid, raw_ptr, bytes;
    cudaIpcMemHandle_t ipc;
};
static_assert(sizeof(TpBlob) <= 256, "blob too large");
static_assert(TOPK_MAX == Q3_TOPK_MAX, "k_topk_logprobs is built for Q3_TOPK_MAX");
extern "C" size_t q3_tp_blob_size(void) { return 256; }

extern "C" int q3_tp_export(q3_handle *h, void *blob_out) {
    if (!h || !blob_out) return fail(Q3_EINVAL, "null argument");
    CK(cudaSetDevice(h->device));
    memset(blob_out, 0, 256);
    TpBlob b{};
    b.magic = 0x51335450; // "Q3TP"
    b.rank = h->tp_rank; b.tp_size = h->tp_size; b.device = h->device;
    b.pid = (uint64_t)getpid();
    b.raw_ptr = (uint64_t)(uintptr_t)h->xchg;
    b.bytes = h->xchg_bytes;
    CK(cudaIpcGetMemHandle(&b.ipc, h->xchg));
    memcpy(blob_out, &b, sizeof b);
    return Q3_OK;
}

extern "C" int q3_tp_connect(q3_handle *h, const void *blobs) {
    if (!h || !blobs) return fail(Q3_EINVAL, "null argument");
    if (h->tp_size == 1) return Q3_OK;
    CK(cudaSetDevice(h->device));
    MegaArgs &a = h->margs;
    for (int r = 0; r < h->tp_size; r++) {
        TpBlob b;
        memcpy(&b, (const uint8_t *)blobs + (size_t)r * 256, sizeof b);
        if (b.magic != 0x51335450 || (int)b.rank != r || (int)b.tp_size != h->tp_size || b.bytes != h->xchg_bytes)
            return fail(Q3_ECOMM, "rank %d: bad exchange blob (rank %u, tp %u, %llu bytes)", r, b.rank, b.tp_size,
                        (unsigned long long)b.bytes);
        uint8_t *base = nullptr;
        if (r == h->tp_rank) {
            base = h->xchg;
        } else if (b.pid == (uint64_t)getpid()) { // same process: plain peer access
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, h->device, (int)b.device));
            if (!can) return fail(Q3_ECOMM, "device %d cannot access peer device %u", h->device, b.device);
            cudaError_t e = cudaDeviceEnablePeerAccess((int)b.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                return fail(Q3_ECOMM, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            cudaGetLastError();
            base = (uint8_t *)(uintptr_t)b.raw_ptr;
        } else { // another process on this node: CUDA IPC over NVLink
            void *p = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&p, b.ipc, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) return fail(Q3_ECOMM, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
            h->peer_maps.push_back(p);
            base = (uint8_t *)p;
        }
        a.part[0][r] = (unsigned long long *)(base + h->off_part[0]);
        a.part[1][r] = (unsigned long long *)(base + h->off_part[1]);
        a.best[r] = (unsigned long long *)(base + h->off_best);
        a.xbar[r] = (unsigned long long *)(base + h->off_flags);
        a.logits[r] = (float *)(base + h->off_logits);
        for (int i = 0; i < 2; i++) {
            h->pf_peers[i].part[r] = (const float *)(base + h->off_pf_part[i]);
            h->pf_peers[i].ctr[r] = (unsigned long long *)(base + h->off_pf_ctr);
        }
    }
    h->tp_connected = true;
    return Q3_OK;
}

extern "C" int q3_tp_set_logits_root(q3_handle *h, int root) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    if (root >= h->tp_size) return fail(Q3_EINVAL, "logits root %d outside the tensor-parallel group of %d", root, h->tp_size);
    h->logits_root = root < 0 ? -1 : root;
    return Q3_OK;
}

extern "C" void q3_destroy(q3_handle *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (int e = 0; e < 32; e++) {
        if (h->g_fwd[e]) cudaGraphExecDestroy(h->g_fwd[e]);
        if (h->g_greedy[e]) cudaGraphExecDestroy(h->g_greedy[e]);
    }
    prefill_release(h);
    if (h->sc_logits) cudaFree(h->sc_logits);
    if (h->tk_ids) cudaFree(h->tk_ids);
    for (void *p : h->peer_maps) cudaIpcCloseMemHandle(p);
    for (void *p : h->allocs) cudaFree(p);
    if (h->h_logits) cudaFreeHost(h->h_logits);
    if (h->h_small) cudaFreeHost(h->h_small);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" const q3_config *q3_get_config(const q3_handle *h) { return h ? &h->cfg : nullptr; }
extern "C" const float *q3_logits_device(const q3_handle *h) { return h ? h->logits : nullptr; }
extern "C" float *q3_logits_host(q3_handle *h) { return h ? h->h_logits : nullptr; }
extern "C" int q3_launches_per_step(const q3_handle *h) { return h ? h->launches_per_step : 0; }
extern "C" int q3_set_decode_path(q3_handle *h, int path) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    if (path != 0 && path != 1) return fail(Q3_EINVAL, "decode path %d unknown", path);
    if (path == 0 && h->tp_size > 1) return fail(Q3_EUNSUPPORTED, "the multi-kernel path has no tensor-parallel exchange");
    if (path == 1 && !h->mega_ok)
        return fail(Q3_EUNSUPPORTED, "persistent decode kernel unavailable for this shape: %s", h->mega_why.c_str());
    h->decode_path = path;
    h->launches_per_step = path == 1 ? 1 : h->graph_launches_per_step;
    return Q3_OK;
}

extern "C" int q3_set_exact_mask(q3_handle *h, int mask) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    if (mask < 0 || mask > 31) return fail(Q3_EINVAL, "exact mask %d outside 0..31", mask);
    CK(cudaSetDevice(h->device));
    if (mask && h->tp_size > 1) return fail(Q3_EUNSUPPORTED, "exact mode is single-GPU");
    if (mask && h->cfg.dim > 16384) return fail(Q3_EUNSUPPORTED, "exact mode needs dim <= 16384");
    h->exact = mask;
    if (!h->g_fwd[h->exact]) return build_graphs(h);
    return Q3_OK;
}
extern "C" int q3_set_exact(q3_handle *h, int on) { return q3_set_exact_mask(h, on ? 31 : 0); }

static int check_tok_pos(const q3_handle *h, int token, int pos) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    if (int rc = tp_ready(h)) return rc;
    if (token < 0 || token >= h->cfg.vocab_size)
        return fail(Q3_EINVAL, "index out of bounds: token %d >= vocab_size %d", token, h->cfg.vocab_size);
    if (pos < 0 || pos >= h->cfg.seq_len)
        return fail(Q3_EINVAL, "index out of bounds: pos %d >= seq_len %d", pos, h->cfg.seq_len);
    return 0;
}

// a prompt of n tokens at positions pos0 .. pos0+n-1 (q3_prefill, q3_bench_prefill, q3_score): the batched path gathers the
// embedding rows of the tokens on the device unchecked
static int check_prompt(const q3_handle *h, const int *tokens, int n, int pos0) {
    if (!h || !tokens || n <= 0) return fail(Q3_EINVAL, "bad prompt arguments");
    if (pos0 < 0 || (long long)pos0 + n > h->cfg.seq_len)
        return fail(Q3_EINVAL, "index out of bounds: pos0 %d + n %d > seq_len %d", pos0, n, h->cfg.seq_len);
    for (int i = 0; i < n; i++)
        if (tokens[i] < 0 || tokens[i] >= h->cfg.vocab_size)
            return fail(Q3_EINVAL, "index out of bounds: token %d >= vocab_size %d", tokens[i], h->cfg.vocab_size);
    if (h->tp_size > 1 && !h->tp_connected) return fail(Q3_ECOMM, "tensor-parallel handle used before q3_tp_connect");
    return 0;
}

static int set_tok_pos(q3_handle *h, int token, int pos) {
    h->h_small[0] = token;
    h->h_small[1] = pos;
    h->h_small[2] = 0;
    h->h_small[3] = 0;
    CK(cudaMemcpyAsync(h->d_tokpos, h->h_small, 16, cudaMemcpyHostToDevice, h->stream));
    return 0;
}

extern "C" int q3_forward(q3_handle *h, int token, int pos, float *logits_host) {
    int rc = check_tok_pos(h, token, pos);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if ((rc = set_tok_pos(h, token, pos))) return rc;
    if (logits_host && h->tp_size > 1 && h->logits_root >= 0 && h->logits_root != h->tp_rank)
        return fail(Q3_EINVAL, "rank %d asked for logits but the logits root is rank %d", h->tp_rank, h->logits_root);
    if ((rc = launch_decode_step(h, STEP_LOGITS, logits_host != nullptr))) return rc;
    if (logits_host) CK(cudaMemcpyAsync(h->h_logits, h->logits, (size_t)h->cfg.vocab_size * 4, cudaMemcpyDeviceToHost, h->stream));
    if ((rc = finish_call(h))) return rc;
    if (logits_host && logits_host != h->h_logits) memcpy(logits_host, h->h_logits, (size_t)h->cfg.vocab_size * 4);
    return Q3_OK;
}

extern "C" int q3_forward_argmax(q3_handle *h, int token, int pos, int *next_token) {
    int rc = check_tok_pos(h, token, pos);
    if (rc) return rc;
    if (!next_token) return fail(Q3_EINVAL, "null next_token");
    CK(cudaSetDevice(h->device));
    if ((rc = set_tok_pos(h, token, pos))) return rc;
    if ((rc = launch_decode_step(h, STEP_FEEDBACK))) return rc;
    CK(cudaMemcpyAsync(h->h_small + 8, h->d_tokpos + 2, 4, cudaMemcpyDeviceToHost, h->stream));
    if ((rc = finish_call(h))) return rc;
    *next_token = h->h_small[8];
    return Q3_OK;
}

extern "C" int q3_decode_greedy(q3_handle *h, int first_token, int pos0, int n, int *tokens_out) {
    int rc = check_tok_pos(h, first_token, pos0);
    if (rc) return rc;
    if (n < 0 || pos0 + n > h->cfg.seq_len) return fail(Q3_EINVAL, "pos0 + n = %d exceeds seq_len %d", pos0 + n, h->cfg.seq_len);
    if (n > h->history_cap) return fail(Q3_EINVAL, "n too large");
    CK(cudaSetDevice(h->device));
    if ((rc = set_tok_pos(h, first_token, pos0))) return rc;
    for (int i = 0; i < n; i++)
        if ((rc = launch_decode_step(h, STEP_FEEDBACK))) return rc;
    if (tokens_out && n > 0) CK(cudaMemcpyAsync(tokens_out, h->d_history, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    return finish_call(h);
}

// ------------------------------------------------------------------------------------------
// device sampler: Sampler::new / sample (sampler.rs:30-41, 116-136)
// ------------------------------------------------------------------------------------------
static size_t next_pow2(size_t n) {
    size_t p = 1;
    while (p < n) p <<= 1;
    return p;
}
extern "C" int q3_sampler_set(q3_handle *h, float temperature, float topp, unsigned long long rng_seed) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    if (!(temperature >= 0.0f)) return fail(Q3_EINVAL, "Temperature must be non-negative");
    if (!(topp >= 0.0f && topp <= 1.0f)) return fail(Q3_EINVAL, "Top-p must be between 0.0 and 1.0");
    CK(cudaSetDevice(h->device));
    int rc;
    if (!h->d_rng) {
        if ((rc = dmalloc(h, (void **)&h->d_rng, 64))) return rc;
        if ((rc = dmalloc(h, (void **)&h->d_probs, (size_t)h->cfg.vocab_size * 4))) return rc;
        if ((rc = dmalloc(h, (void **)&h->d_keys, next_pow2((size_t)h->cfg.vocab_size) * 8))) return rc;
    }
    h->samp_temperature = temperature;
    h->samp_topp = topp;
    CK(cudaMemcpyAsync(h->d_rng, &rng_seed, 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return Q3_OK;
}
extern "C" int q3_sampler_state(q3_handle *h, unsigned long long *rng_state_out) {
    if (!h || !rng_state_out) return fail(Q3_EINVAL, "null argument");
    if (!h->d_rng) return fail(Q3_EINVAL, "q3_sampler_set has not been called");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(rng_state_out, h->d_rng, 8, cudaMemcpyDeviceToHost));
    return Q3_OK;
}
extern "C" int q3_sampler_skip(q3_handle *h, int n_draws) {
    if (!h || n_draws < 0) return fail(Q3_EINVAL, "bad argument");
    if (!h->d_rng) return fail(Q3_EINVAL, "q3_sampler_set has not been called");
    CK(cudaSetDevice(h->device));
    if (h->samp_temperature != 0.0f && n_draws > 0) k_rng_skip<<<1, 1, 0, h->stream>>>(h->d_rng, n_draws); // greedy draws no coin (:117-119)
    CK(cudaGetLastError());
    return Q3_OK;
}
// one decode step + sample on the device; feedback: the sampled token / next position stay on the device for the next step
static int launch_sampled_step(q3_handle *h, bool feedback) {
    int rc;
    const bool greedy = h->samp_temperature == 0.0f;
    // greedy: the step's own argmax; otherwise k_sample draws from the full logits
    if ((rc = launch_decode_step(h, !greedy ? STEP_LOGITS : feedback ? STEP_FEEDBACK : STEP_ARGMAX, !greedy))) return rc;
    if (!greedy) {
        SampleArgs a{};
        a.logits = h->logits; a.n = h->cfg.vocab_size; a.temperature = h->samp_temperature; a.topp = h->samp_topp;
        a.rng_state = h->d_rng; a.p = h->d_probs; a.keys = h->d_keys; a.token_out = h->d_tokpos + 2;
        if (feedback) { a.token_feedback = h->d_tokpos; a.pos_advance = h->d_tokpos + 1; a.history = h->d_history; a.history_idx = h->d_tokpos + 3; }
        k_sample<<<1, SAMPLE_THREADS, 0, h->stream>>>(a);
        CK(cudaGetLastError());
    }
    return 0;
}
extern "C" int q3_forward_sample(q3_handle *h, int token, int pos, int *next_token) {
    int rc = check_tok_pos(h, token, pos);
    if (rc) return rc;
    if (!next_token) return fail(Q3_EINVAL, "null next_token");
    if (!h->d_rng) return fail(Q3_EINVAL, "q3_sampler_set has not been called");
    CK(cudaSetDevice(h->device));
    if ((rc = set_tok_pos(h, token, pos))) return rc;
    if ((rc = launch_sampled_step(h, false))) return rc;
    CK(cudaMemcpyAsync(h->h_small + 8, h->d_tokpos + 2, 4, cudaMemcpyDeviceToHost, h->stream));
    if ((rc = finish_call(h))) return rc;
    *next_token = h->h_small[8];
    return Q3_OK;
}
extern "C" int q3_decode_sample(q3_handle *h, int first_token, int pos0, int n, int *tokens_out) {
    int rc = check_tok_pos(h, first_token, pos0);
    if (rc) return rc;
    if (n < 0 || pos0 + n > h->cfg.seq_len) return fail(Q3_EINVAL, "pos0 + n = %d exceeds seq_len %d", pos0 + n, h->cfg.seq_len);
    if (n > h->history_cap) return fail(Q3_EINVAL, "n too large");
    if (!h->d_rng) return fail(Q3_EINVAL, "q3_sampler_set has not been called");
    CK(cudaSetDevice(h->device));
    if ((rc = set_tok_pos(h, first_token, pos0))) return rc;
    for (int i = 0; i < n; i++)
        if ((rc = launch_sampled_step(h, true))) return rc;
    if (tokens_out && n > 0) CK(cudaMemcpyAsync(tokens_out, h->d_history, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    return finish_call(h);
}

extern "C" int q3_bench_decode(q3_handle *h, int first_token, int pos0, int steps, float *ms_out) {
    int rc = check_tok_pos(h, first_token, pos0);
    if (rc) return rc;
    if (steps < 1 || pos0 + steps > h->cfg.seq_len) return fail(Q3_EINVAL, "pos0 + steps exceeds seq_len");
    CK(cudaSetDevice(h->device));
    if ((rc = set_tok_pos(h, first_token, pos0))) return rc;
    float ms = 0;
    rc = time_events(h->stream, &ms, [&] {
        for (int i = 0; i < steps; i++)
            if (int rc1 = launch_decode_step(h, STEP_FEEDBACK)) return rc1;
        return 0;
    });
    if (rc) return rc;
    if (ms_out) *ms_out = ms;
    return finish_call(h);
}

extern "C" int q3_bench_kernel(q3_handle *h, int kind, int pos, int reps, float *ms_out, int *launches_out,
                               double *bytes_out) {
    if (!h || kind < 0 || kind > 5 || reps < 1) return fail(Q3_EINVAL, "bad bench arguments");
    if (pos < 0 || pos >= h->cfg.seq_len) return fail(Q3_EINVAL, "index out of bounds: pos %d", pos);
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = set_tok_pos(h, 0, pos))) return rc;
    const q3_config &c = h->cfg;
    const int gs = c.group_size, ns = h->num_sms, ex = h->exact, dim = c.dim, L = c.n_layers;
    auto one = [&](int l) {
        const LayerDev &W = h->layers[l];
        float *kc_l = h->kc + (size_t)l * c.seq_len * h->KV_l;
        float *vc_l = h->vc + (size_t)l * c.seq_len * h->KV_l;
        GemvArgs g{};
        g.xq = h->xq; g.xs = h->xs; g.pos = h->d_tokpos + 1;
        switch (kind) {
        case 0:
            g.wq = W.qkv.q; g.ws = W.qkv.s; g.K = dim; g.rows = W.qkv.rows; g.q = h->q; g.kc = kc_l; g.vc = vc_l;
            g.AH = h->AH_l; g.KV = h->KV_l;
            launch_gemv<EPI_QKV>(gs, ns, ex, g, h->stream);
            break;
        case 1:
            g.wq = W.wo.q; g.ws = W.wo.s; g.K = h->AH_l; g.rows = dim; g.out = h->xb;
            launch_gemv<EPI_STORE>(gs, ns, ex, g, h->stream);
            break;
        case 2:
            g.wq = W.w13.q; g.ws = W.w13.s; g.K = dim; g.rows = W.w13.rows; g.out = h->hb;
            launch_gemv<EPI_SWIGLU>(gs, ns, ex, g, h->stream);
            break;
        case 3:
            g.wq = W.w2.q; g.ws = W.w2.s; g.xq = h->hq; g.xs = h->hs; g.K = h->H_l; g.rows = dim; g.out = h->xb;
            launch_gemv<EPI_STORE>(gs, ns, ex, g, h->stream);
            break;
        case 4:
            g.wq = h->wcls.q; g.ws = h->wcls.s; g.K = dim; g.rows = c.vocab_size; g.out = h->logits;
            launch_gemv<EPI_STORE>(gs, ns, ex, g, h->stream);
            break;
        case 5:
            launch_attn_partial(h, kc_l, vc_l, h->stream);
            break;
        }
    };
    double bytes = 0;
    const double sc = 1.0 + 4.0 / gs;
    switch (kind) {
    case 0: bytes = (double)h->layers[0].qkv.rows * dim * sc; break;
    case 1: bytes = (double)dim * h->AH_l * sc; break;
    case 2: bytes = (double)h->layers[0].w13.rows * dim * sc; break;
    case 3: bytes = (double)dim * h->H_l * sc; break;
    case 4: bytes = (double)c.vocab_size * dim * sc; break;
    case 5: bytes = 2.0 * (pos + 1) * h->KV_l * 4; break;
    }
    for (int l = 0; l < L; l++) one(l); // warm-up pass
    float ms = 0;
    rc = time_events(h->stream, &ms, [&] {
        for (int r = 0; r < reps; r++)
            for (int l = 0; l < L; l++) one(l);
        return 0;
    });
    if (rc) return rc;
    if (ms_out) *ms_out = ms;
    if (launches_out) *launches_out = reps * L;
    if (bytes_out) *bytes_out = bytes;
    return Q3_OK;
}

extern "C" int q3_prefill(q3_handle *h, const int *tokens, int n, int pos0, float *last_logits_host) {
    if (int rc = check_prompt(h, tokens, n, pos0)) return rc;
    CK(cudaSetDevice(h->device));
    if (!h->pf_ok || h->exact) {
        // sequential decode steps: same results as n forwards by construction (exact mode, TP, odd shapes)
        for (int i = 0; i < n; i++) {
            int rc = q3_forward(h, tokens[i], pos0 + i, i == n - 1 ? last_logits_host : nullptr);
            if (rc) return rc;
        }
        return Q3_OK;
    }
    int rc;
    if ((rc = prefill_chunks(h, tokens, n, pos0))) return rc;
    // final norm + quantize + lm_head on the last token only (qwen3.rs:72-76)
    if ((rc = set_tok_pos(h, tokens[n - 1], pos0 + n - 1))) return rc;
    if ((rc = launch_head_only(h, last_logits_host != nullptr))) return rc;
    if (last_logits_host) CK(cudaMemcpyAsync(h->h_logits, h->logits, (size_t)h->cfg.vocab_size * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaGetLastError());
    if ((rc = finish_call(h))) return rc;
    if (last_logits_host && last_logits_host != h->h_logits) memcpy(last_logits_host, h->h_logits, (size_t)h->cfg.vocab_size * 4);
    return Q3_OK;
}

extern "C" int q3_bench_prefill(q3_handle *h, const int *tokens, int n, int pos0, float *ms_out) {
    int rc = check_prompt(h, tokens, n, pos0);
    if (rc) return rc;
    if (!h->pf_ok) return fail(Q3_EUNSUPPORTED, "batched prefill unavailable: %s", h->pf_why.c_str());
    CK(cudaSetDevice(h->device));
    if ((rc = prefill_chunks(h, tokens, n, pos0))) return rc; // warm-up (also sizes the buffers)
    float ms = 0;
    if ((rc = time_events(h->stream, &ms, [&] { return prefill_chunks(h, tokens, n, pos0); }))) return rc;
    if (ms_out) *ms_out = ms;
    return finish_call(h);
}

// q3_score (k 0) and q3_score_topk (k 1 .. Q3_TOPK_MAX, ids / lps required)
static int score_impl(q3_handle *h, const int *tokens, int n, int pos0, int k, int *ids_out, float *lps_out, const int *targets,
                      float *logprobs_out, int *argmax_out) {
    int rc = check_prompt(h, tokens, n, pos0);
    if (rc) return rc;
    if (k) {
        if (k < 1 || k > Q3_TOPK_MAX || k > h->cfg.vocab_size)
            return fail(Q3_EINVAL, "k %d outside 1 .. min(%d, vocab %d)", k, Q3_TOPK_MAX, h->cfg.vocab_size);
        if (!ids_out || !lps_out) return fail(Q3_EINVAL, "q3_score_topk needs topk_ids_out and topk_logprobs_out");
    } else if (!logprobs_out && !argmax_out) {
        return fail(Q3_EINVAL, "q3_score needs logprobs_out or argmax_out");
    }
    if (logprobs_out && !targets) return fail(Q3_EINVAL, "logprobs_out needs targets");
    const int V = h->cfg.vocab_size;
    if (logprobs_out)
        for (int i = 0; i < n; i++)
            if (targets[i] < 0 || targets[i] >= V) return fail(Q3_EINVAL, "index out of bounds: target %d", targets[i]);
    const bool batched = h->pf_ok && !h->exact && V % 128 == 0;
    // Under TP, q3_forward leaves only this rank's vocabulary shard in h->logits (all of it only on the logits root, if one is set)
    if (h->tp_size > 1 && !batched) return fail(Q3_EUNSUPPORTED, "q3_score under tensor parallelism needs the batched prefill path");
    CK(cudaSetDevice(h->device));
    if ((rc = score_reserve(h, batched, n))) return rc;
    if (k && (rc = topk_reserve(h, k))) return rc;
    h->sc_want_lp = logprobs_out != nullptr;
    h->tk_k = k;
    if (logprobs_out) CK(cudaMemcpyAsync(h->sc_targets, targets, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
    if (batched) {
        if ((rc = prefill_chunks(h, tokens, n, pos0, true))) return rc;
    } else {
        // sequential decode steps (exact mode: the logits are the reference's bit for bit), reduced one at a time
        for (int i = 0; i < n; i++) {
            if ((rc = q3_forward(h, tokens[i], pos0 + i, nullptr))) return rc;
            launch_logprobs(h, h->logits, 1, i);
        }
    }
    if (logprobs_out) CK(cudaMemcpyAsync(logprobs_out, h->sc_lp, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (argmax_out) CK(cudaMemcpyAsync(argmax_out, h->sc_argmax, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    if (k) {
        CK(cudaMemcpyAsync(ids_out, h->tk_ids, (size_t)n * k * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(lps_out, h->tk_lps, (size_t)n * k * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaGetLastError());
    return finish_call(h);
}

extern "C" int q3_score(q3_handle *h, const int *tokens, int n, int pos0, const int *targets, float *logprobs_out, int *argmax_out) {
    return score_impl(h, tokens, n, pos0, 0, nullptr, nullptr, targets, logprobs_out, argmax_out);
}

extern "C" int q3_score_topk(q3_handle *h, const int *tokens, int n, int pos0, int k, int *topk_ids_out, float *topk_logprobs_out,
                             const int *targets, float *logprobs_out, int *argmax_out) {
    if (k == 0) return fail(Q3_EINVAL, "k must be at least 1"); // k 0 selects q3_score's path in score_impl
    return score_impl(h, tokens, n, pos0, k, topk_ids_out, topk_logprobs_out, targets, logprobs_out, argmax_out);
}

extern "C" int q3_reset(q3_handle *h) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    CK(cudaSetDevice(h->device));
    size_t kvn = (size_t)h->cfg.n_layers * h->cfg.seq_len * h->KV_l;
    CK(cudaMemsetAsync(h->kc, 0, kvn * 4, h->stream));
    CK(cudaMemsetAsync(h->vc, 0, kvn * 4, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return Q3_OK;
}

static int kv_rw(q3_handle *h, int layer, int pos0, int n, float *k, float *v, bool write) {
    if (!h) return fail(Q3_EINVAL, "null handle");
    if (layer < 0 || layer >= h->cfg.n_layers || pos0 < 0 || n < 0 || pos0 + n > h->cfg.seq_len)
        return fail(Q3_EINVAL, "kv range out of bounds");
    CK(cudaSetDevice(h->device));
    size_t off = ((size_t)layer * h->cfg.seq_len + pos0) * h->KV_l, bytes = (size_t)n * h->KV_l * 4;
    cudaMemcpyKind kind = write ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    CK(cudaStreamSynchronize(h->stream));
    if (k) CK(write ? cudaMemcpy(h->kc + off, k, bytes, kind) : cudaMemcpy(k, h->kc + off, bytes, kind));
    if (v) CK(write ? cudaMemcpy(h->vc + off, v, bytes, kind) : cudaMemcpy(v, h->vc + off, bytes, kind));
    return Q3_OK;
}
extern "C" int q3_kv_read(q3_handle *h, int layer, int pos0, int n, float *k, float *v) {
    return kv_rw(h, layer, pos0, n, k, v, false);
}
extern "C" int q3_kv_write(q3_handle *h, int layer, int pos0, int n, const float *k, const float *v) {
    return kv_rw(h, layer, pos0, n, (float *)k, (float *)v, true);
}

extern "C" int q3_forward_layers(q3_handle *h, int pos, int layer0, int layer1, float *x_host, int run_head,
                                 float *logits_host) {
    if (!h || !x_host) return fail(Q3_EINVAL, "null argument");
    if (pos < 0 || pos >= h->cfg.seq_len) return fail(Q3_EINVAL, "index out of bounds: pos %d", pos);
    if (layer0 < 0 || layer1 > h->cfg.n_layers || layer0 > layer1) return fail(Q3_EINVAL, "bad layer range");
    CK(cudaSetDevice(h->device));
    int rc;
    if ((rc = tp_ready(h))) return rc;
    if ((rc = set_tok_pos(h, 0, pos))) return rc;
    CK(cudaMemcpyAsync(h->x, x_host, (size_t)h->cfg.dim * 4, cudaMemcpyHostToDevice, h->stream));
    if (use_mega(h)) {
        if (layer1 > layer0 && (rc = launch_mega(h, layer0, layer1, false, false, false, false))) return rc;
    } else {
        for (int l = layer0; l < layer1; l++) launch_layer(h, l, false, h->stream);
    }
    CK(cudaMemcpyAsync(x_host, h->x, (size_t)h->cfg.dim * 4, cudaMemcpyDeviceToHost, h->stream));
    if (run_head) {
        if ((rc = launch_head_only(h, true))) return rc;
        if (logits_host)
            CK(cudaMemcpyAsync(logits_host, h->logits, (size_t)h->cfg.vocab_size * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaGetLastError());
    return finish_call(h);
}

// ------------------------------------------------------------------------------------------
// operator-level entry points
// ------------------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
    int alloc(size_t n) { CK(cudaMalloc(&p, n ? n : 16)); return 0; }
    template <class T> T *as() { return (T *)p; }
};
static int op_prologue(int device, int gs) {
    CK(cudaSetDevice(device));
    if (gs != 32 && gs != 64 && gs != 128) return fail(Q3_EUNSUPPORTED, "group_size %d unsupported (32/64/128)", gs);
    return 0;
}

extern "C" int q3_op_quantize(int device, const float *x, int n, int gs, int8_t *q_out, float *s_out) {
    int rc = op_prologue(device, gs);
    if (rc) return rc;
    if (n < 0 || n % gs) return fail(Q3_EINVAL, "n must be a multiple of group_size");
    if (n == 0) return Q3_OK;
    DevBuf dx, dq, ds;
    if ((rc = dx.alloc((size_t)n * 4)) || (rc = dq.alloc(n)) || (rc = ds.alloc((size_t)n / gs * 4))) return rc;
    CK(cudaMemcpy(dx.p, x, (size_t)n * 4, cudaMemcpyHostToDevice));
    int grid = (n / 4 + 255) / 256;
    GS_DISPATCH(gs, (k_quantize<GS><<<grid, 256>>>(dx.as<float>(), n, dq.as<int8_t>(), ds.as<float>())));
    CK(cudaGetLastError());
    CK(cudaMemcpy(q_out, dq.p, n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(s_out, ds.p, (size_t)n / gs * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

__global__ void k_expf_ref(const float *x, float *out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = expf_ref(x[i]);
}
extern "C" int q3_op_expf(int device, const float *x, int n, float *out) {
    CK(cudaSetDevice(device));
    if (n <= 0) return Q3_OK;
    DevBuf dx, dout;
    int rc;
    if ((rc = dx.alloc((size_t)n * 4)) || (rc = dout.alloc((size_t)n * 4))) return rc;
    CK(cudaMemcpy(dx.p, x, (size_t)n * 4, cudaMemcpyHostToDevice));
    k_expf_ref<<<(n + 255) / 256, 256>>>(dx.as<float>(), dout.as<float>(), n);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

extern "C" int q3_op_matmul(int device, const int8_t *xq, const float *xs, const int8_t *wq, const float *ws, int n,
                            int d, int gs, int exact, float *out, int32_t *group_dots_out) {
    int rc = op_prologue(device, gs);
    if (rc) return rc;
    if (n <= 0 || d < 0 || n % gs || n % 16 || d % 2) return fail(Q3_EINVAL, "need n %% gs == 0, n %% 16 == 0, d even");
    if (d == 0) return Q3_OK;
    const int ng = n / gs;
    DevBuf dxq, dxs, dwq, dws, dout, ddots;
    if ((rc = dxq.alloc(n)) || (rc = dxs.alloc((size_t)ng * 4)) || (rc = dwq.alloc((size_t)d * n)) ||
        (rc = dws.alloc((size_t)d * ng * 4)) || (rc = dout.alloc((size_t)d * 4)))
        return rc;
    if (group_dots_out && (rc = ddots.alloc((size_t)d * ng * 4))) return rc;
    CK(cudaMemcpy(dxq.p, xq, n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dxs.p, xs, (size_t)ng * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dwq.p, wq, (size_t)d * n, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dws.p, ws, (size_t)d * ng * 4, cudaMemcpyHostToDevice));
    GemvArgs a{};
    a.wq = dwq.as<int8_t>(); a.ws = dws.as<float>(); a.xq = dxq.as<int8_t>(); a.xs = dxs.as<float>();
    a.K = n; a.rows = d; a.out = dout.as<float>(); a.dots = group_dots_out ? ddots.as<int32_t>() : nullptr;
    int num_sms = 0;
    CK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));
    if ((rc = prepare_exact_kernels())) return rc;
    launch_gemv<EPI_STORE>(gs, num_sms, exact ? 31 : 0, a, 0);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout.p, (size_t)d * 4, cudaMemcpyDeviceToHost));
    if (group_dots_out) CK(cudaMemcpy(group_dots_out, ddots.p, (size_t)d * ng * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

extern "C" int q3_op_gemm_q8(int device, const int8_t *xq, const float *xs, const int8_t *wq, const float *ws, int T, int N,
                             int K, int gs, int exact, float *out) {
    int rc = op_prologue(device, gs);
    if (rc) return rc;
    if (T <= 0 || N % 128 || K % 128 || K % gs || (K / gs) % 2) return fail(Q3_EINVAL, "need N %% 128 == 0, K %% 128 == 0 and an even number of groups per row");
    if (exact != 0 && exact != 1) return fail(Q3_EINVAL, "exact must be 0 (fast drain) or 1 (exact drain), not %d", exact);
    const int Tpad = (T + 127) / 128 * 128, ng = K / gs;
    DevBuf dxq, dxsT, dwq, dws, dwsT, dout;
    if ((rc = dxq.alloc((size_t)Tpad * K)) || (rc = dxsT.alloc((size_t)ng * Tpad * 4)) || (rc = dwq.alloc((size_t)N * K)) ||
        (rc = dws.alloc((size_t)N * ng * 4)) || (rc = dwsT.alloc((size_t)N * ng * 4)) || (rc = dout.alloc((size_t)Tpad * N * 4)))
        return rc;
    // output sentinel: every byte 0xFF (a NaN) -- an element the kernel skips reads back as NaN, and the padding rows past T,
    // which the epilogue must never store, are checked below
    CK(cudaMemset(dout.p, 0xFF, (size_t)Tpad * N * 4));
    CK(cudaMemset(dxq.p, 0, (size_t)Tpad * K));
    CK(cudaMemcpy(dxq.p, xq, (size_t)T * K, cudaMemcpyHostToDevice));
    std::vector<float> xsT((size_t)ng * Tpad, 0.0f);
    for (int t = 0; t < T; t++)
        for (int g = 0; g < ng; g++) xsT[(size_t)g * Tpad + t] = xs[(size_t)t * ng + g];
    CK(cudaMemcpy(dxsT.p, xsT.data(), xsT.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dwq.p, wq, (size_t)N * K, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dws.p, ws, (size_t)N * ng * 4, cudaMemcpyHostToDevice));
    dim3 tg((ng + 31) / 32, (N + 31) / 32);
    k_transpose_f32<<<tg, dim3(32, 8)>>>(dws.as<float>(), dwsT.as<float>(), N, ng);
    CUtensorMap mx, mw;
    if ((rc = make_map_i8(&mx, dxq.p, Tpad, K)) || (rc = make_map_i8(&mw, dwq.p, N, K))) return rc;
    PrefillGemmArgs a{};
    a.T = T; a.Tpad = Tpad; a.N = N; a.K = K; a.wsT = dwsT.as<float>(); a.xsT = dxsT.as<float>(); a.out = dout.as<float>(); a.ld_out = N;
    if ((rc = launch_gemm_q8<PF_EPI_STORE>(gs, mx, mw, a, 0, exact))) return rc;
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out, dout.p, (size_t)T * N * 4, cudaMemcpyDeviceToHost));
    std::vector<uint32_t> pad((size_t)(Tpad - T) * N);
    if (!pad.empty()) {
        CK(cudaMemcpy(pad.data(), dout.as<float>() + (size_t)T * N, pad.size() * 4, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < pad.size(); i++)
            if (pad[i] != 0xFFFFFFFFu)
                return fail(Q3_ECUDA, "GEMM wrote padding row %d (T %d) at column %d", T + (int)(i / N), T, (int)(i % N));
    }
    return Q3_OK;
}

// Sampler::sample on host-supplied logits (operator-level parity entry): one draw, RNG state in / out
extern "C" int q3_op_sample(int device, const float *logits, int n, float temperature, float topp, unsigned long long *rng_state,
                            int *token_out) {
    CK(cudaSetDevice(device));
    if (!logits || !rng_state || !token_out || n <= 0) return fail(Q3_EINVAL, "bad argument");
    if (!(temperature > 0.0f)) return fail(Q3_EINVAL, "temperature must be positive (0 = greedy: use the argmax path)");
    DevBuf dl, dp, dk, dr, dt;
    int rc;
    if ((rc = dl.alloc((size_t)n * 4)) || (rc = dp.alloc((size_t)n * 4)) || (rc = dk.alloc(next_pow2((size_t)n) * 8)) || (rc = dr.alloc(8)) ||
        (rc = dt.alloc(4)))
        return rc;
    CK(cudaMemcpy(dl.p, logits, (size_t)n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dr.p, rng_state, 8, cudaMemcpyHostToDevice));
    SampleArgs a{};
    a.logits = dl.as<float>(); a.n = n; a.temperature = temperature; a.topp = topp < 0.f ? 0.f : (topp > 1.f ? 1.f : topp);
    a.rng_state = dr.as<unsigned long long>(); a.p = dp.as<float>(); a.keys = dk.as<unsigned long long>(); a.token_out = dt.as<int>();
    k_sample<<<1, SAMPLE_THREADS>>>(a);
    CK(cudaGetLastError());
    CK(cudaMemcpy(rng_state, dr.p, 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(token_out, dt.p, 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

// q3_score's reduction on host-supplied logits [rows][n]: log-softmax at targets[r] and the last argmax of every row
extern "C" int q3_op_logprobs(int device, const float *logits, int rows, int n, const int *targets, float *logprobs_out, int *argmax_out) {
    if (!logits || rows <= 0 || n <= 0) return fail(Q3_EINVAL, "bad logprobs arguments");
    if (!logprobs_out && !argmax_out) return fail(Q3_EINVAL, "q3_op_logprobs needs logprobs_out or argmax_out");
    if (logprobs_out && !targets) return fail(Q3_EINVAL, "logprobs_out needs targets");
    if (logprobs_out)
        for (int r = 0; r < rows; r++)
            if (targets[r] < 0 || targets[r] >= n) return fail(Q3_EINVAL, "index out of bounds: target %d (n %d)", targets[r], n);
    CK(cudaSetDevice(device));
    DevBuf dl, dt, dlp, dam;
    int rc;
    if ((rc = dl.alloc((size_t)rows * n * 4)) || (rc = dt.alloc((size_t)rows * 4)) || (rc = dlp.alloc((size_t)rows * 4)) ||
        (rc = dam.alloc((size_t)rows * 4)))
        return rc;
    CK(cudaMemcpy(dl.p, logits, (size_t)rows * n * 4, cudaMemcpyHostToDevice));
    if (logprobs_out) CK(cudaMemcpy(dt.p, targets, (size_t)rows * 4, cudaMemcpyHostToDevice));
    k_logprobs<<<rows, LP_THREADS>>>(dl.as<float>(), n, (size_t)n, dt.as<int>(), logprobs_out ? dlp.as<float>() : nullptr, dam.as<int>());
    CK(cudaGetLastError());
    if (logprobs_out) CK(cudaMemcpy(logprobs_out, dlp.p, (size_t)rows * 4, cudaMemcpyDeviceToHost));
    if (argmax_out) CK(cudaMemcpy(argmax_out, dam.p, (size_t)rows * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

// q3_score_topk's reduction on host-supplied logits [rows][n]: the k largest entries of every row (descending value, ties to
// the larger index) with their log-softmax, and optionally q3_op_logprobs' two outputs from the same pass
extern "C" int q3_op_topk_logprobs(int device, const float *logits, int rows, int n, int k, const int *targets, int *ids_out,
                                   float *lps_out, float *logprobs_out, int *argmax_out) {
    if (!logits || rows <= 0 || n <= 0) return fail(Q3_EINVAL, "bad top-k arguments");
    if (k < 1 || k > Q3_TOPK_MAX || k > n) return fail(Q3_EINVAL, "k %d outside 1 .. min(%d, n %d)", k, Q3_TOPK_MAX, n);
    if (!ids_out || !lps_out) return fail(Q3_EINVAL, "q3_op_topk_logprobs needs ids_out and lps_out");
    if (logprobs_out && !targets) return fail(Q3_EINVAL, "logprobs_out needs targets");
    if (logprobs_out)
        for (int r = 0; r < rows; r++)
            if (targets[r] < 0 || targets[r] >= n) return fail(Q3_EINVAL, "index out of bounds: target %d (n %d)", targets[r], n);
    CK(cudaSetDevice(device));
    DevBuf dl, dt, dlp, dam, di, dv;
    int rc;
    const size_t rk = (size_t)rows * k;
    if ((rc = dl.alloc((size_t)rows * n * 4)) || (rc = dt.alloc((size_t)rows * 4)) || (rc = dlp.alloc((size_t)rows * 4)) ||
        (rc = dam.alloc((size_t)rows * 4)) || (rc = di.alloc(rk * 4)) || (rc = dv.alloc(rk * 4)))
        return rc;
    CK(cudaMemcpy(dl.p, logits, (size_t)rows * n * 4, cudaMemcpyHostToDevice));
    if (logprobs_out) CK(cudaMemcpy(dt.p, targets, (size_t)rows * 4, cudaMemcpyHostToDevice));
    k_topk_logprobs<<<rows, LP_THREADS>>>(dl.as<float>(), n, (size_t)n, k, di.as<int>(), dv.as<float>(), dt.as<int>(),
                                          logprobs_out ? dlp.as<float>() : nullptr, argmax_out ? dam.as<int>() : nullptr);
    CK(cudaGetLastError());
    CK(cudaMemcpy(ids_out, di.p, rk * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(lps_out, dv.p, rk * 4, cudaMemcpyDeviceToHost));
    if (logprobs_out) CK(cudaMemcpy(logprobs_out, dlp.p, (size_t)rows * 4, cudaMemcpyDeviceToHost));
    if (argmax_out) CK(cudaMemcpy(argmax_out, dam.p, (size_t)rows * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

// Causal prefill attention alone (layers.rs:374-419 for T query tokens at positions pos0 .. pos0+T-1 over a cache of pos0+T rows):
// q [T][n_heads*128] (already normalised + rotated), k / v [pos0+T][n_kv*128], out [T][n_heads*128].
// The launch is the one q3_prefill runs (launch_pf_attention: k_pf_attention_h over a hi / lo split of K / V).
extern "C" int q3_op_prefill_attention(int device, const float *q, const float *k, const float *v, int T, int pos0, int n_heads, int n_kv,
                                       float *out) {
    CK(cudaSetDevice(device));
    if (!q || !k || !v || !out || T <= 0 || pos0 < 0 || n_kv <= 0 || n_heads % n_kv) return fail(Q3_EINVAL, "bad attention arguments");
    const int kv_mul = n_heads / n_kv;
    if (kv_mul != 1 && kv_mul != 2 && kv_mul != 4 && kv_mul != 8) return fail(Q3_EUNSUPPORTED, "GQA factor %d unsupported", kv_mul);
    const int AH = n_heads * HEAD_DIM, KV = n_kv * HEAD_DIM, nk = pos0 + T;
    DevBuf dq, dk, dv, dout, dkvh;
    int rc;
    if ((rc = dq.alloc((size_t)T * AH * 4)) || (rc = dk.alloc((size_t)nk * KV * 4)) || (rc = dv.alloc((size_t)nk * KV * 4)) ||
        (rc = dout.alloc((size_t)T * AH * 4)) || (rc = dkvh.alloc((size_t)4 * nk * KV * 2)))
        return rc;
    CK(cudaMemcpy(dq.p, q, (size_t)T * AH * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dk.p, k, (size_t)nk * KV * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dv.p, v, (size_t)nk * KV * 4, cudaMemcpyHostToDevice));
    int num_sms = 0;
    CK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device));
    if ((rc = allow_pf_attention(kv_mul))) return rc;
    launch_pf_attention(dq.as<float>(), dk.as<float>(), dv.as<float>(), dkvh.as<__half>(), (size_t)nk * KV, dout.as<float>(), T, pos0, n_kv,
                        kv_mul, num_sms, 0);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out, dout.p, (size_t)T * AH * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

// Timing helper: the tcgen05 GEMM alone on device-resident random operands, CUDA events; mode as in q3_op_gemm_q8
// (0 fast drain, 1 exact drain).  ms_out = milliseconds per launch (best of reps).
__global__ void k_fill_i8(int8_t *p, size_t n, unsigned seed) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        unsigned h = (unsigned)i * 2654435761u + seed;
        h ^= h >> 15;
        p[i] = (int8_t)((h * 2246822519u >> 24) - 128);
    }
}
__global__ void k_fill_f32(float *p, size_t n, float v) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
extern "C" int q3_bench_gemm_q8(int device, int T, int N, int K, int gs, int mode, int reps, float *ms_out) {
    int rc = op_prologue(device, gs);
    if (rc) return rc;
    if (T <= 0 || N % 128 || K % 128 || K % gs || (K / gs) % 2 || reps < 1 || (mode != 0 && mode != 1)) return fail(Q3_EINVAL, "bad gemm bench arguments");
    const int Tpad = (T + 127) / 128 * 128, ng = K / gs;
    DevBuf dxq, dxsT, dwq, dwsT, dout;
    if ((rc = dxq.alloc((size_t)Tpad * K)) || (rc = dxsT.alloc((size_t)ng * Tpad * 4)) || (rc = dwq.alloc((size_t)N * K)) ||
        (rc = dwsT.alloc((size_t)N * ng * 4)) || (rc = dout.alloc((size_t)T * N * 4)))
        return rc;
    k_fill_i8<<<592, 256>>>(dxq.as<int8_t>(), (size_t)Tpad * K, 1);
    k_fill_i8<<<592, 256>>>(dwq.as<int8_t>(), (size_t)N * K, 2);
    k_fill_f32<<<592, 256>>>(dxsT.as<float>(), (size_t)ng * Tpad, 0.01f);
    k_fill_f32<<<592, 256>>>(dwsT.as<float>(), (size_t)N * ng, 0.02f);
    CUtensorMap mx, mw;
    if ((rc = make_map_i8(&mx, dxq.p, Tpad, K)) || (rc = make_map_i8(&mw, dwq.p, N, K))) return rc;
    PrefillGemmArgs a{};
    a.T = T; a.Tpad = Tpad; a.N = N; a.K = K; a.wsT = dwsT.as<float>(); a.xsT = dxsT.as<float>(); a.out = dout.as<float>(); a.ld_out = N;
    if ((rc = launch_gemm_q8<PF_EPI_STORE>(gs, mx, mw, a, 0, mode))) return rc; // warm-up
    CK(cudaDeviceSynchronize());
    float best = 1e30f;
    for (int r = 0; r < reps; r++) {
        float ms = 0;
        if ((rc = time_events(0, &ms, [&] { return launch_gemm_q8<PF_EPI_STORE>(gs, mx, mw, a, 0, mode); }))) return rc;
        best = ms < best ? ms : best;
    }
    if (ms_out) *ms_out = best;
    return Q3_OK;
}

extern "C" int q3_op_rmsnorm(int device, const float *x, const float *w, int n, float *out) {
    CK(cudaSetDevice(device));
    if (n <= 0) return fail(Q3_EINVAL, "n must be positive");
    DevBuf dx, dw, dout;
    int rc;
    if ((rc = dx.alloc((size_t)n * 4)) || (rc = dw.alloc((size_t)n * 4)) || (rc = dout.alloc((size_t)n * 4))) return rc;
    CK(cudaMemcpy(dx.p, x, (size_t)n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(dw.p, w, (size_t)n * 4, cudaMemcpyHostToDevice));
    k_rmsnorm<<<1, 1024>>>(dx.as<float>(), dw.as<float>(), dout.as<float>(), n);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, dout.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}

// same kernel on buffers that already live on the device (bench / fixture generation of multi-GB checkpoints)
extern "C" int q3_op_quantize_q80_dev(int device, const float *w_dev, size_t n, int gs, int8_t *q_dev, float *s_dev) {
    int rc = op_prologue(device, gs);
    if (rc) return rc;
    if (n % gs) return fail(Q3_EINVAL, "Weight length is not a multiple of group_size");
    if (n == 0) return Q3_OK;
    if (!w_dev || !q_dev || !s_dev) return fail(Q3_EINVAL, "null argument");
    size_t blocks = (n / 4 + 255) / 256;
    int grid = (int)(blocks > 148 * 16 ? 148 * 16 : blocks);
    GS_DISPATCH(gs, (k_quantize_q80<GS><<<grid, 256>>>(w_dev, n, q_dev, s_dev)));
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return Q3_OK;
}

extern "C" int q3_op_quantize_q80(int device, const float *w, size_t n, int gs, int8_t *q_out, float *s_out) {
    int rc = op_prologue(device, gs);
    if (rc) return rc;
    if (n % gs) return fail(Q3_EINVAL, "Weight length is not a multiple of group_size");
    if (n == 0) return Q3_OK;
    DevBuf dw, dq, ds;
    if ((rc = dw.alloc(n * 4)) || (rc = dq.alloc(n)) || (rc = ds.alloc(n / gs * 4))) return rc;
    CK(cudaMemcpy(dw.p, w, n * 4, cudaMemcpyHostToDevice));
    size_t blocks = (n / 4 + 255) / 256;
    int grid = (int)(blocks > 148 * 16 ? 148 * 16 : blocks);
    GS_DISPATCH(gs, (k_quantize_q80<GS><<<grid, 256>>>(dw.as<float>(), n, dq.as<int8_t>(), ds.as<float>())));
    CK(cudaGetLastError());
    CK(cudaMemcpy(q_out, dq.p, n, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(s_out, ds.p, n / gs * 4, cudaMemcpyDeviceToHost));
    return Q3_OK;
}
