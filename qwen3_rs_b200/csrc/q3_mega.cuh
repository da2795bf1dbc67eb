// q3_mega.cuh -- persistent single-launch decode step ("megakernel") for sm_100a.
//
// One cooperative launch per token: 148 CTAs (one per SM) walk the whole forward pass
// (qwen3.rs:62-79, 131-176) phase by phase.  Inside each CTA two PRODUCER threads (one per
// consumer group) stream the CTA's share of the int8 weights HBM -> shared memory with
// cp.async.bulk (TMA, 1-D) into a 4-stage ring of mbarrier-guarded stages, and run AHEAD of the
// consumers across phase and layer boundaries (weights do not depend on activations), so HBM
// stays busy while the 16 CONSUMER warps (two groups owning alternate stages) wait on a
// dependency or rebuild the quantised activation vector.  Consumers keep their slice of the
// activation vector in registers and do the int8 dot products with dp4a out of shared memory.
// The K/V cache rows an attention CTA needs travel through the SAME ring (2-D TMA tiles of 32 positions,
// issued by the producers right behind the QKV weights): they are in shared memory before the
// attention step starts, and at long context the cache streams at HBM rate instead of at the rate
// register-held loads can sustain.
//
// Dependencies: there is NO grid barrier inside a layer.  Every datum that crosses CTAs travels as a
// 64-bit (payload, epoch) word (see ll_store) that its consumer polls:
//   qkv rows          -> zone Q, polled by the (kv head, split) attention CTAs (only the rows of their kv group)
//   attention output  -> merged, normalised and QUANTISED once by the last-arriving split of a kv head, published
//                        as packed int8 + scales in zone A (already in the o_proj shared-memory order)
//   o_proj / down     -> zone O / D (under tensor parallelism: partial rows pushed into every peer GPU over NVLink,
//                        reduced once by the CTA that owns the row, republished locally)
//   SwiGLU outputs    -> zone H, quantised by every CTA for down_proj
// The only grid barrier left is the one before the greedy argmax (one per token).
//
// HBM "stream" layout (built once at load by k_build_stream): for every GEMV phase, rows are
// split contiguously over CTAs; a CTA's rows are stored in the exact order its consumers eat
// them, one "row tile" (KT <= 4096 columns + their f32 scales) per consumer warp per stage,
// and inside a tile the 16-byte chunks are permuted so that lane l owns whole quantisation
// groups (l, l+32, ...) while every 128-bit shared-memory load stays bank-conflict free.
//
// Float semantics are those of the fast multi-kernel path (q3_kernels.cuh): identical per-group
// terms, parallel reductions.  Exact (reference-order) mode uses the multi-kernel path.
#pragma once
#include <cuda.h>

#include "q3_kernels.cuh"

namespace q3 {

#ifndef MEGA_GW_
#define MEGA_GW_ 8
#endif
constexpr int MEGA_GW = MEGA_GW_;                    // consumer warps per group = row tiles per stage
constexpr int MEGA_BATCH = 4 * MEGA_GW;             // rows per batch of a row phase (up to 4 stages per K tile)
constexpr int MEGA_GROUPS = 2;                      // consumer groups; stages alternate between them
constexpr int MEGA_NCW = MEGA_GW * MEGA_GROUPS;     // 16 consumer warps
constexpr int MEGA_CTHREADS = MEGA_NCW * 32;        // 512 consumer threads
// + one producer warp per consumer group.  (A producer warpgroup that hands its registers to the consumers with
// setmaxnreg was tried: ptxas cannot allocate this kernel's consumer path in 112-120 registers without spilling and
// refuses -- see DESIGN.md.)
constexpr int MEGA_THREADS = MEGA_CTHREADS + 32 * MEGA_GROUPS;
#ifndef MEGA_NSTAGE_
#define MEGA_NSTAGE_ 4
#endif
constexpr int MEGA_NSTAGE = MEGA_NSTAGE_;
constexpr int MEGA_MAX_KT = 4096;
constexpr int MEGA_SCRATCH = 40960;                 // xq/xs or attention buffers
constexpr int MEGA_MAX_TP = 8;
constexpr int MEGA_MAX_SPLITS = ATTN_MAX_SPLITS;
constexpr int MEGA_EDGES = 6;                       // epochs per layer: one per step kind (0 qkv .. 4 down), one spare; the head step uses the next layer's 0

enum { PH_QKV = 0, PH_O = 1, PH_GU = 2, PH_DN = 3, PH_HEAD = 4 };

struct MegaGemv {
    const uint8_t *base;     // stream of layer 0 (or the lm_head stream)
    long long layer_stride;  // bytes between layers
    int units;               // rows, or (gate, up) PAIRS for PH_GU
    int K, n_kt, KT, G;      // columns, K tiles per row, columns per tile, groups per tile
    int tile_bytes;          // KT + 4*G rounded up to 16 B (bulk copies move 16-byte units)
};

constexpr int MEGA_KV_ROWS = 32; // cache positions per K/V stage (= MEGA_ATTN_CHUNK): 32 x 512 B of K + 32 x 512 B of V

struct MegaArgs {
    // TMA descriptors of the K and V caches seen as 2-D f32 tensors [n_layers * seq_len rows][KV_l], box = 32 rows x 128 floats:
    // one bulk-tensor copy brings 32 consecutive positions of one kv head (16 KB) into a ring stage
    alignas(64) CUtensorMap map_k;
    alignas(64) CUtensorMap map_v;
    int dim, n_layers, n_heads_l, n_kv_l, AH_l, KV_l, H_l, vocab_l, vocab_row0, seq_len;
    int tp_rank, tp_size;
    MegaGemv g[5];
    const float *rms_att, *rms_ffn, *q_ln, *k_ln, *rms_final; // [L][dim] / [L][128] contiguous
    const int8_t *embed_q;
    const float *embed_s;
    const float *rope;
    float *kc, *vc;
    float *x;                        // residual stream in / out of a teacher-forced layer range (read-only in a head-only launch)
    // (payload, epoch) zones, all zero-initialised; see ll_store
    unsigned long long *zq;          // [AH_l + 2 KV_l]        q | k | v rows of the current layer (raw GEMV results)
    unsigned long long *za;          // [AH_l/4 + AH_l/GS]     quantised attention output (4 int8 per word, PH_O smem order) | group scales
    unsigned long long *zh;          // [H_l]                  SwiGLU outputs
    unsigned long long *zr[2];       // [dim]                  o_proj / down rows, reduced over the TP ranks (this rank's copy)
    unsigned long long *part[2][MEGA_MAX_TP]; // TP only: [o|down][rank] -> that rank's landing zone [tp][dim] (peer memory)
    float *attn_part;                // [n_heads_l][MEGA_MAX_SPLITS][ATTN_PART_STRIDE] split partials (nsplit > 1)
    unsigned *att_cnt;               // [n_layers][n_kv_l] arrivals of the splits of a kv head (returns to 0 within the launch)
    float *logits[MEGA_MAX_TP];      // full-vocab logits buffer of every rank
    unsigned long long *best[MEGA_MAX_TP]; // [tp][grid] argmax candidates of every rank
    unsigned long long *bar;         // grid barrier counter (monotonic, never reset)
    unsigned long long bar_base;     // counter value when this launch starts (host-tracked)
    unsigned long long *xbar[MEGA_MAX_TP]; // cross-GPU barrier counter of every rank (peer memory under TP)
    unsigned long long xbar_base;    // value of the cross counters when this launch starts (host-tracked)
    int *tokpos, *history;
    int *status;                     // != 0: a wait timed out (kernel aborts)
    int layer0, layer1, from_embed, run_head, feedback, gather_logits;
    unsigned ll_base;                // epoch counter before this launch, already reduced mod 2^32 - 1 (host-tracked, same on every TP rank)
    unsigned long long *prof;        // optional [grid][MEGA_PROF_EVENTS] clock64 stamps (thread 0 of each CTA)
};
// In-kernel profiler: thread 0 of every CTA appends (clock64 << 8 | tag).  Tags: 0 start; 1 + 3*kind + {0 prologue done,
// 1 GEMV done, 2 step-end sync done} for step kinds 0..5; >= 32 finer marks inside the prologues and the grid barrier.
// The last slot of a CTA's row holds its event count.
constexpr int MEGA_PROF_EVENTS = 4096;
struct Prof {
    unsigned long long *row;
    int ev;
};
#define prof_mark(p, tag)                                                                                              \
    do {                                                                                                               \
        if (a.prof) { /* kernel parameter (constant bank): the Prof struct is not touched unless a capture is running */ \
            Prof &p_ = (p);                                                                                            \
            if (p_.row && p_.ev < MEGA_PROF_EVENTS - 1) p_.row[p_.ev++] = ((unsigned long long)clock64() << 8) | (unsigned)(tag); \
        }                                                                                                              \
    } while (0)

// ------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + bulk copy
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return ok != 0;
}
// Waits never hang the GPU: after ~2 s (a scheduling bug, not a stall) the waiter raises the abort
// flag (device memory, polled only every 4096 spins) and everybody falls through.
__device__ __noinline__ void mbar_wait_slow(uint64_t *bar, uint32_t parity, int *status);
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity, int *status) {
    if (mbar_try_wait(bar, parity)) return; // common case: already complete, no call
    mbar_wait_slow(bar, parity, status);
}
__device__ __noinline__ void mbar_wait_slow(uint64_t *bar, uint32_t parity, int *status) {
    long long t0 = clock64();
    unsigned spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 4095u) == 0) {
            if (*(volatile int *)status) return;
            if (clock64() - t0 > 4000000000LL) {
                atomicExch(status, 2);
                return;
            }
        }
    }
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int c0, int c1, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, %0;" ::"n"(MEGA_CTHREADS) : "memory"); }
__device__ __forceinline__ float ldcg_f(const float *p) { return __ldcg(p); }
__device__ __forceinline__ float4 ldcg_f4(const float *p) { return __ldcg(reinterpret_cast<const float4 *>(p)); }

// ------------------------------------------------------------------------------------------
// (payload, epoch) words: a 64-bit store is single-copy atomic, so a reader that sees the expected epoch in the upper half
// holds the payload that was written with it -- no fence on the writer, no barrier between writer and reader (the NCCL "LL"
// idea, here for every cross-CTA edge of a layer, and across GPUs over NVLink peer stores).
// Why nothing else is needed:
//  * the words are the ONLY data that crosses CTAs inside a layer (the residual stream lives in each CTA's shared
//    memory; the attention split partials are ordered by a fence + counter, see attention_item);
//  * epochs are unique per (launch, layer, edge): a host-tracked counter, the same sequence on every TP rank, reduced
//    mod 2^32 - 1 and offset by 1 so that 0 (the zero-initialised zones) is never a valid epoch and wrap-around is harmless
//    (a zone is completely rewritten at every use, so a stale word is always exactly one use old);
//  * a zone is rewritten one layer later.  A writer gets there only after it has consumed words of later edges that every
//    CTA (every CTA of every rank) produces only after it has finished reading the previous contents: every CTA owns at
//    least one qkv row and one gate/up unit (checked at load), all qkv rows are polled by some attention CTA, and zones
//    A / O / H / D are polled completely by every CTA (argument per zone in DESIGN.md section 4).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned ll_epoch(unsigned base, unsigned k) {
    unsigned long long s = (unsigned long long)base + k;
    if (s >= 0xFFFFFFFFull) s -= 0xFFFFFFFFull;
    return (unsigned)s + 1u;
}
__device__ __forceinline__ void ll_store_u32(unsigned long long *p, unsigned payload, unsigned epoch) {
    const unsigned long long w = ((unsigned long long)epoch << 32) | (unsigned long long)payload;
    asm volatile("st.relaxed.sys.global.b64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ void ll_store(unsigned long long *p, float v, unsigned epoch) { ll_store_u32(p, __float_as_uint(v), epoch); }
__device__ __forceinline__ void ll_load2(const unsigned long long *p, unsigned long long &x, unsigned long long &y) {
    asm volatile("ld.relaxed.sys.global.v2.b64 {%0,%1}, [%2];" : "=l"(x), "=l"(y) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned long long ll_load1(const unsigned long long *p) {
    unsigned long long x;
    asm volatile("ld.relaxed.sys.global.b64 %0, [%1];" : "=l"(x) : "l"(p) : "memory");
    return x;
}
__device__ __forceinline__ bool ll_ok(unsigned long long w, unsigned epoch) { return (unsigned)(w >> 32) == epoch; }
// called after a failed poll: give up (abort flag, status `code`) after ~1-2 s -- a protocol bug must never hang the GPU
__device__ __noinline__ bool ll_give_up(const MegaArgs &a, unsigned &spins, int code) {
    if ((++spins & 255u) == 0) {
        if (*(volatile int *)a.status) return true;
        if (spins > (1u << 20)) {
            atomicExch(a.status, code);
            return true;
        }
    }
    return false;
}
// poll 4 consecutive words (16-byte aligned pair of pairs) and return their payloads as a float4
__device__ __forceinline__ float4 ll_poll4(const MegaArgs &a, const unsigned long long *p, unsigned epoch, int code) {
    unsigned long long w0, w1, w2, w3;
    unsigned spins = 0;
    while (true) {
        ll_load2(p, w0, w1);
        ll_load2(p + 2, w2, w3);
        if (ll_ok(w0, epoch) && ll_ok(w1, epoch) && ll_ok(w2, epoch) && ll_ok(w3, epoch)) break;
        if (ll_give_up(a, spins, code)) break;
    }
    return make_float4(__uint_as_float((unsigned)w0), __uint_as_float((unsigned)w1), __uint_as_float((unsigned)w2), __uint_as_float((unsigned)w3));
}

// contiguous split of `units` over `nctas`
__device__ __host__ __forceinline__ void cta_share(int units, int nctas, int c, int &start, int &count) {
    int base = units / nctas, rem = units % nctas;
    count = base + (c < rem ? 1 : 0);
    start = c * base + (c < rem ? c : rem);
}

// ------------------------------------------------------------------------------------------
// stream builder: row-major int8 [rows][K] + scales [rows][K/GS]  ->  megakernel stream
// grid = (units, n_kt); one block per unit (row, or gate/up pair) and K tile.
// ------------------------------------------------------------------------------------------
template <int GS>
__global__ void __launch_bounds__(256) k_build_stream(const int8_t *__restrict__ src_q, const float *__restrict__ src_s,
                                                      uint8_t *dst, int units, int K, int n_kt, int nctas, int pair) {
    constexpr int CPG = GS / 16;
    const int u = blockIdx.x, kt = blockIdx.y;
    const int KT = K / n_kt, G = KT / GS, tile_bytes = KT + ((4 * G + 15) & ~15); // scale area padded to 16 B
    const int base = units / nctas, rem = units % nctas;
    int c, j;
    if (u < rem * (base + 1)) {
        c = u / (base + 1);
        j = u % (base + 1);
    } else {
        c = rem + (u - rem * (base + 1)) / base;
        j = (u - rem * (base + 1)) % base;
    }
    int start, n_c;
    cta_share(units, nctas, c, start, n_c);
    for (int half = 0; half < (pair ? 2 : 1); half++) {
        long long tile_index;
        size_t src_row;
        if (pair) { // blocks of MEGA_GW pairs: [gate x np][up x np]
            int blk = j / MEGA_GW, w = j % MEGA_GW, np = n_c - MEGA_GW * blk;
            if (np > MEGA_GW) np = MEGA_GW;
            tile_index = (long long)start * 2 + 2 * MEGA_GW * blk + half * np + w;
            src_row = (size_t)2 * u + half;
        } else { // batches of 32 rows: [kt][row]
            int b = j / MEGA_BATCH, jb = j % MEGA_BATCH, nb = n_c - MEGA_BATCH * b;
            if (nb > MEGA_BATCH) nb = MEGA_BATCH;
            tile_index = ((long long)start + MEGA_BATCH * b) * n_kt + (long long)kt * nb + jb;
            src_row = (size_t)u;
        }
        uint8_t *tile = dst + tile_index * tile_bytes;
        const int8_t *srow = src_q + src_row * K + (size_t)kt * KT;
        for (int ch = threadIdx.x; ch < KT / 16; ch += blockDim.x) {
            int g = ch / CPG, p = ch % CPG, b = g / 32, l = g % 32;
            int ngb = G - 32 * b;
            if (ngb > 32) ngb = 32;
            int dpos = b * 32 * CPG + p * ngb + l;
            reinterpret_cast<int4 *>(tile)[dpos] = reinterpret_cast<const int4 *>(srow)[ch];
        }
        const float *ss = src_s + src_row * (K / GS) + (size_t)kt * G;
        for (int g = threadIdx.x; g < G; g += blockDim.x) reinterpret_cast<float *>(tile + KT)[g] = ss[g];
    }
}

// ------------------------------------------------------------------------------------------
// consumer-side building blocks
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int4 lds128(uint32_t saddr) {
    int4 r;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(saddr));
    return r;
}
__device__ __forceinline__ float lds_f32(uint32_t saddr) {
    float r;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(r) : "r"(saddr));
    return r;
}
template <int GS>
struct XRegs { // this lane's groups of the current K tile: MEGA_MAX_KT/128 = 32 registers + scales
    static constexpr int CPG = GS / 16;
    static constexpr int NBLK = MEGA_MAX_KT / (32 * GS);
    int4 x[NBLK][CPG];
    float s[NBLK];
};

// The quantised activation sits in shared memory in the SAME chunk permutation as a weight row tile
// (lane l owns groups l, l+32, ...; its 16-byte chunks are 16*ngb bytes apart), so the 128-bit loads
// below are conflict-free.  (Element order would put consecutive lanes GS bytes apart: a 16-way bank
// conflict -- ~1 us per call with 16 warps, 7 calls per layer.)
// byte offset of float4 #i4 of the activation vector inside the (K-tiled, chunk-permuted) shared-memory image
template <int GS>
__device__ __forceinline__ int xq_offset(int i4, int KT, int G) {
    int r = i4 * 4, off = 0;
    while (r >= KT) { // K tile (at most 4)
        r -= KT;
        off += KT;
    }
    const int g = r / GS, b = g >> 5, l = g & 31;
    int ngb = G - 32 * b;
    ngb = ngb > 32 ? 32 : ngb;
    const int p = (r % GS) >> 4;
    return off + b * 32 * GS + (p * ngb + l) * 16 + (r & 15);
}
template <int GS>
__device__ __forceinline__ void xq_store(uint8_t *sxq, int i4, uint32_t packed, int KT, int G) {
    *reinterpret_cast<uint32_t *>(sxq + xq_offset<GS>(i4, KT, G)) = packed;
}
template <int GS>
__device__ __forceinline__ void load_x(XRegs<GS> &xr, const uint8_t *sxq, const float *sxs, int kt, int KT, int G, int lane) {
    const uint32_t base = smem_u32(sxq) + kt * KT + lane * 16;
#pragma unroll
    for (int b = 0; b < XRegs<GS>::NBLK; b++) {
        int ngb = G - 32 * b;
        ngb = ngb > 32 ? 32 : ngb;
        const bool ok = lane < ngb;
        if (ngb < 1) ngb = 1;
        xr.s[b] = ok ? sxs[kt * G + b * 32 + lane] : 0.0f;
#pragma unroll
        for (int p = 0; p < XRegs<GS>::CPG; p++)
            xr.x[b][p] = ok ? lds128(base + b * 32 * GS + p * ngb * 16) : make_int4(0, 0, 0, 0);
    }
}

// dot of one row tile (in shared memory) with the register-resident activation slice.
// Per group: exact int32 dot, then (dot as f32 * weight_scale) * input_scale (tensor.rs:47-59).
// All 128-bit shared loads of the tile are issued before the first dp4a (explicit ld.shared.v4:
// left to itself the compiler split them into 32-bit loads under the 96-register cap), and each
// block runs two independent dp4a chains.  FULL: every block has 32 groups (G % 32 == 0), so all
// offsets are immediates and no lane is predicated off.
template <int GS, bool FULL>
__device__ __forceinline__ float tile_dot(uint32_t tile, const XRegs<GS> &xr, int KT, int G, int lane) {
    constexpr int CPG = XRegs<GS>::CPG;
    constexpr int NBLK = XRegs<GS>::NBLK;
    int4 w[NBLK][CPG];
    float ws[NBLK];
#pragma unroll
    for (int b = 0; b < NBLK; b++) {
        int ngb = FULL ? 32 : (G - 32 * b > 32 ? 32 : G - 32 * b);
        const bool on = FULL ? (32 * b < G) : (lane < ngb);
        if (!FULL && ngb < 1) ngb = 1;
        const uint32_t base = tile + b * 32 * GS + lane * 16;
#pragma unroll
        for (int p = 0; p < CPG; p++) w[b][p] = on ? lds128(base + p * ngb * 16) : make_int4(0, 0, 0, 0);
        ws[b] = on ? lds_f32(tile + KT + (b * 32 + lane) * 4) : 0.0f;
    }
    float acc = 0.0f;
#pragma unroll
    for (int b = 0; b < NBLK; b++) {
        int d0 = 0, d1 = 0; // two independent dp4a chains; int32 addition is exact in any order
#pragma unroll
        for (int p = 0; p < CPG; p += 2) {
            d0 = dot16(w[b][p], xr.x[b][p], d0);
            d1 = dot16(w[b][p + 1], xr.x[b][p + 1], d1);
        }
        acc = __fadd_rn(acc, __fmul_rn(__fmul_rn((float)(d0 + d1), ws[b]), xr.s[b]));
    }
    return warp_sum(acc);
}

// RMSNorm + group quantise of the residual stream into shared memory (all 512 consumer threads).
// Also adds the result of the previous row-parallel GEMV (o_proj / down_proj: x <- x + row, ResidualConnection
// layers.rs:249-259; under TP the row is already the rank-ordered sum of the partials, see the reduce step in the kernel,
// so every rank computes bit-identical x) and gathers the embedding row.
constexpr int MEGA_MAXV = (MEGA_MAX_KT + 4 * MEGA_CTHREADS - 1) / (4 * MEGA_CTHREADS); // float4 per thread of a dim <= 4096 vector

// src: 0 = embedding row of tokpos[0], 1 = a.x (teacher-forced entry), 2 = sx (this CTA's copy of the residual stream in
// shared memory; a thread always owns the same elements).  zone/epoch: pending GEMV rows to add (or null).
template <int GS>
__device__ __noinline__ void prologue_norm(const MegaArgs &a, const float *w, int src, const unsigned long long *zone, unsigned epoch,
                                           uint8_t *sxq, float *sxs, float *sred, float *sx, int KT, int G, Prof &pr) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n4 = a.dim >> 2;
    constexpr int MAXV = MEGA_MAXV;
    float4 v[MAXV], wv[MAXV];
    float ss = 0.0f;
    // the norm weights do not depend on the activation: with the weight stream saturating the memory system a global
    // round trip costs ~1.3 us, so their loads are issued before the poll below instead of after it
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        const int i4 = tid + k * MEGA_CTHREADS;
        wv[k] = (i4 < n4) ? __ldg(reinterpret_cast<const float4 *>(w) + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        const int i4 = tid + k * MEGA_CTHREADS;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i4 < n4) {
            if (src == 0) {
                size_t base = (size_t)a.tokpos[0] * a.dim + (size_t)i4 * 4;
                char4 e = *reinterpret_cast<const char4 *>(a.embed_q + base);
                float sc = a.embed_s[base / GS];
                v[k] = make_float4((float)e.x * sc, (float)e.y * sc, (float)e.z * sc, (float)e.w * sc);
            } else if (src == 1) {
                v[k] = ldcg_f4(a.x + (size_t)i4 * 4);
            } else {
                v[k] = reinterpret_cast<const float4 *>(sx)[i4];
            }
        }
    }
    if (zone) { // every word is taken as soon as it carries `epoch`; all loads of a thread are in flight together
        unsigned long long ww[MAXV][4];
        unsigned spins = 0;
        while (true) {
            bool ok = true;
#pragma unroll
            for (int k = 0; k < MAXV; k++) {
                const int i4 = tid + k * MEGA_CTHREADS;
                if (i4 < n4) {
                    ll_load2(zone + (size_t)i4 * 4, ww[k][0], ww[k][1]);
                    ll_load2(zone + (size_t)i4 * 4 + 2, ww[k][2], ww[k][3]);
                    ok = ok && ll_ok(ww[k][0], epoch) && ll_ok(ww[k][1], epoch) && ll_ok(ww[k][2], epoch) && ll_ok(ww[k][3], epoch);
                }
            }
            if (ok || ll_give_up(a, spins, 6)) break;
        }
#pragma unroll
        for (int k = 0; k < MAXV; k++) {
            if (tid + k * MEGA_CTHREADS < n4) {
                v[k].x = __fadd_rn(v[k].x, __uint_as_float((unsigned)ww[k][0]));
                v[k].y = __fadd_rn(v[k].y, __uint_as_float((unsigned)ww[k][1]));
                v[k].z = __fadd_rn(v[k].z, __uint_as_float((unsigned)ww[k][2]));
                v[k].w = __fadd_rn(v[k].w, __uint_as_float((unsigned)ww[k][3]));
            }
        }
    }
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        const int i4 = tid + k * MEGA_CTHREADS;
        if (i4 < n4) {
            reinterpret_cast<float4 *>(sx)[i4] = v[k];
            ss += __fmul_rn(v[k].x, v[k].x);
            ss += __fmul_rn(v[k].y, v[k].y);
            ss += __fmul_rn(v[k].z, v[k].z);
            ss += __fmul_rn(v[k].w, v[k].w);
        }
    }
    prof_mark(pr, 32); // x (+ pending rows) arrived
    ss = warp_sum(ss);
    if (lane == 0) sred[warp] = ss;
    csync(); // also: every warp has left the previous GEMV, sxq may be rewritten
    float t = 0.0f;
#pragma unroll
    for (int i = 0; i < MEGA_NCW; i++) t += sred[i];
    const float f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(t, (float)a.dim), NORM_EPS)));
    prof_mark(pr, 33); // sum of squares reduced
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        int i4 = tid + k * MEGA_CTHREADS;
        if (i4 - lane < n4) {
            float4 y = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i4 < n4) {
                y.x = __fmul_rn(wv[k].x, __fmul_rn(f, v[k].x));
                y.y = __fmul_rn(wv[k].y, __fmul_rn(f, v[k].y));
                y.z = __fmul_rn(wv[k].z, __fmul_rn(f, v[k].z));
                y.w = __fmul_rn(wv[k].w, __fmul_rn(f, v[k].w));
            }
            uint32_t packed;
            float scale;
            quantize_group4<GS>(y, packed, scale);
            if (i4 < n4) {
                xq_store<GS>(sxq, i4, packed, KT, G);
                if ((i4 % (GS / 4)) == 0) sxs[i4 / (GS / 4)] = scale;
                // (the reference's final norm is in place, qwen3.rs:72, but nothing reads x after it; writing it back from one CTA
                // would race with the other CTAs still reading a.x in a head-only launch)
            }
        }
    }
    prof_mark(pr, 34); // quantised
    csync();
}

// o_proj input: the attention output arrives already normalised and quantised (attention_item), packed 4 int8 per word in the
// chunk order of this phase's shared-memory activation, followed by the group scales -- the prologue is a polled copy.
template <int GS>
__device__ __noinline__ void prologue_attn_poll(const MegaArgs &a, unsigned epoch, uint8_t *sxq, float *sxs) {
    const int tid = threadIdx.x;
    const int nq = a.AH_l >> 2, ng = a.AH_l / GS; // nq is a multiple of 32
    unsigned spins = 0;
    for (int i = 2 * tid; i < nq; i += 2 * MEGA_CTHREADS) {
        unsigned long long x, y;
        while (true) {
            ll_load2(a.za + i, x, y);
            if ((ll_ok(x, epoch) && ll_ok(y, epoch)) || ll_give_up(a, spins, 7)) break;
        }
        *reinterpret_cast<uint2 *>(sxq + 4 * i) = make_uint2((unsigned)x, (unsigned)y);
    }
    for (int g = tid; g < ng; g += MEGA_CTHREADS) {
        unsigned long long x;
        while (true) {
            x = ll_load1(a.za + nq + g);
            if (ll_ok(x, epoch) || ll_give_up(a, spins, 7)) break;
        }
        sxs[g] = __uint_as_float((unsigned)x);
    }
    csync();
}

// down_proj input: poll the SwiGLU outputs (zone H) and group-quantise them into shared memory (layers.rs:478).
// The loads of the next float4 of a thread are in flight while the current one is checked and quantised.
template <int GS>
__device__ __forceinline__ void quant_ll_one(const MegaArgs &a, const unsigned long long *z, unsigned epoch, int i4, int n4, unsigned long long (&w)[4],
                                             unsigned &spins, uint8_t *sxq, float *sxs, int KT, int G) {
    float4 y = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i4 < n4) {
        while (!(ll_ok(w[0], epoch) && ll_ok(w[1], epoch) && ll_ok(w[2], epoch) && ll_ok(w[3], epoch))) {
            if (ll_give_up(a, spins, 8)) break;
            ll_load2(z + (size_t)i4 * 4, w[0], w[1]);
            ll_load2(z + (size_t)i4 * 4 + 2, w[2], w[3]);
        }
        y = make_float4(__uint_as_float((unsigned)w[0]), __uint_as_float((unsigned)w[1]), __uint_as_float((unsigned)w[2]), __uint_as_float((unsigned)w[3]));
    }
    uint32_t packed;
    float scale;
    quantize_group4<GS>(y, packed, scale); // warp-collective: the caller's loop condition is warp-uniform
    if (i4 < n4) {
        xq_store<GS>(sxq, i4, packed, KT, G);
        if ((i4 % (GS / 4)) == 0) sxs[i4 / (GS / 4)] = scale;
    }
}
template <int GS>
__device__ __noinline__ void prologue_quant_ll(const MegaArgs &a, const unsigned long long *z, unsigned epoch, int n, uint8_t *sxq, float *sxs, int KT, int G) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int n4 = n >> 2;
    unsigned long long wa[4] = {0, 0, 0, 0}, wb[4] = {0, 0, 0, 0};
    unsigned spins = 0;
    int i4 = tid;
    if (i4 < n4) {
        ll_load2(z + (size_t)i4 * 4, wa[0], wa[1]);
        ll_load2(z + (size_t)i4 * 4 + 2, wa[2], wa[3]);
    }
#pragma unroll 1
    while (i4 - lane < n4) {
        int j4 = i4 + MEGA_CTHREADS;
        if (j4 < n4) {
            ll_load2(z + (size_t)j4 * 4, wb[0], wb[1]);
            ll_load2(z + (size_t)j4 * 4 + 2, wb[2], wb[3]);
        }
        quant_ll_one<GS>(a, z, epoch, i4, n4, wa, spins, sxq, sxs, KT, G);
        i4 = j4;
        if (!(i4 - lane < n4)) break;
        j4 = i4 + MEGA_CTHREADS;
        if (j4 < n4) {
            ll_load2(z + (size_t)j4 * 4, wa[0], wa[1]);
            ll_load2(z + (size_t)j4 * 4 + 2, wa[2], wa[3]);
        }
        quant_ll_one<GS>(a, z, epoch, i4, n4, wb, spins, sxq, sxs, KT, G);
        i4 = j4;
    }
    csync();
}

// QK-RMSNorm + RoPE of one head held as float4 per lane (same math as k_qknorm_rope); wv = this lane's norm weights,
// cs01 / cs23 = (cos, sin) of its four rotation pairs
__device__ __forceinline__ float4 qk_norm_rope_pre(float4 v, float4 wv, float4 cs01, float4 cs23, int lane) {
    float ss = __fmul_rn(v.x, v.x);
    ss = __fadd_rn(ss, __fmul_rn(v.y, v.y));
    ss = __fadd_rn(ss, __fmul_rn(v.z, v.z));
    ss = __fadd_rn(ss, __fmul_rn(v.w, v.w));
    ss = warp_sum(ss);
    const float f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(ss, (float)HEAD_DIM), NORM_EPS)));
    float4 y;
    y.x = __fmul_rn(wv.x, __fmul_rn(f, v.x));
    y.y = __fmul_rn(wv.y, __fmul_rn(f, v.y));
    y.z = __fmul_rn(wv.z, __fmul_rn(f, v.z));
    y.w = __fmul_rn(wv.w, __fmul_rn(f, v.w));
    float4 o;
    o.x = __shfl_xor_sync(0xffffffffu, y.x, 16);
    o.y = __shfl_xor_sync(0xffffffffu, y.y, 16);
    o.z = __shfl_xor_sync(0xffffffffu, y.z, 16);
    o.w = __shfl_xor_sync(0xffffffffu, y.w, 16);
    float4 r;
    if (lane < 16) {
        r.x = __fsub_rn(__fmul_rn(y.x, cs01.x), __fmul_rn(o.x, cs01.y));
        r.y = __fsub_rn(__fmul_rn(y.y, cs01.z), __fmul_rn(o.y, cs01.w));
        r.z = __fsub_rn(__fmul_rn(y.z, cs23.x), __fmul_rn(o.z, cs23.y));
        r.w = __fsub_rn(__fmul_rn(y.w, cs23.z), __fmul_rn(o.w, cs23.w));
    } else {
        r.x = __fadd_rn(__fmul_rn(o.x, cs01.y), __fmul_rn(y.x, cs01.x));
        r.y = __fadd_rn(__fmul_rn(o.y, cs01.w), __fmul_rn(y.y, cs01.z));
        r.z = __fadd_rn(__fmul_rn(o.z, cs23.y), __fmul_rn(y.z, cs23.x));
        r.w = __fadd_rn(__fmul_rn(o.w, cs23.w), __fmul_rn(y.w, cs23.z));
    }
    return r;
}
__device__ __forceinline__ float4 qk_norm_rope(float4 v, const float *w, const float *rope_row, int lane) {
    const float4 wv = __ldg(reinterpret_cast<const float4 *>(w) + lane);
    const float4 *cs = reinterpret_cast<const float4 *>(rope_row) + (lane & 15) * 2;
    return qk_norm_rope_pre(v, wv, __ldg(cs), __ldg(cs + 1), lane);
}

#ifndef MEGA_ATTN_CHUNK_
#define MEGA_ATTN_CHUNK_ 32
#endif
constexpr int MEGA_ATTN_CHUNK = MEGA_ATTN_CHUNK_; // positions per split before another CTA is recruited
__device__ __forceinline__ int mega_nsplit(int pos, int n_kv_l, int grid) {
    int n = pos + 1;
    int ns = (n + MEGA_ATTN_CHUNK - 1) / MEGA_ATTN_CHUNK;
    int cap = grid / n_kv_l;
    if (cap > MEGA_MAX_SPLITS) cap = MEGA_MAX_SPLITS;
    if (cap < 1) cap = 1;
    return ns > cap ? cap : ns;
}

// normalise (softmax multiplies by 1/sum, layers.rs:504-505), group-quantise (qwen3.rs:152) and publish the 128 outputs of
// one query head held as float4 per lane: packed int8 into zone A at the word the o_proj phase's shared-memory layout
// puts them, scales behind.  Warp-collective.
template <int GS>
__device__ __forceinline__ void publish_head(const MegaArgs &a, int head, int lane, float4 A, float L, unsigned epoch) {
    const float inv = __fdiv_rn(1.0f, L);
    const float4 y = make_float4(__fmul_rn(A.x, inv), __fmul_rn(A.y, inv), __fmul_rn(A.z, inv), __fmul_rn(A.w, inv));
    uint32_t packed;
    float qscale;
    quantize_group4<GS>(y, packed, qscale);
    const int i4 = head * 32 + lane;
    ll_store_u32(a.za + (xq_offset<GS>(i4, a.g[PH_O].KT, a.g[PH_O].G) >> 2), packed, epoch);
    if ((i4 % (GS / 4)) == 0) ll_store(a.za + (a.AH_l >> 2) + i4 / (GS / 4), qscale, epoch);
}

// attention phase for one (kv head, split) work item; all 512 consumer threads.
//   * q (and, in the split that owns `pos`, the new k / v rows) are polled from zone Q -- only this kv group's rows, so the
//     item starts as soon as THEY are done, not when the whole grid is; QK-norm + RoPE (layers.rs:346-372); the owner split
//     stores the k / v cache rows (layers.rs:335-336);
//   * positions t0..t1 with an online softmax (layers.rs:374-419), warp partials merged through shared memory;
//   * one split: normalise + quantise + publish straight away.  Several splits: partials go to global memory, the split that
//     arrives LAST at its kv head's counter merges them, and publishes (release: bar.sync + thread 0's fence before its
//     atomic; acquire: fence after it).
// ring-side state of a consumer warp (see the kernel): stage counter, parities of its group's full barriers
struct RingPos {
    unsigned it, fullp;
};
__device__ __forceinline__ void gsync(int grp) { // the 8 warps of one consumer group
    asm volatile("bar.sync %0, %1;" ::"r"(2 + grp), "n"(MEGA_GW * 32) : "memory");
}

template <int GS, int KVMUL>
__device__ __forceinline__ void attention_item(const MegaArgs &a, int layer, int pos, int kvh, int split, int nsplit,
                                               uint8_t *scratch, unsigned ep_q, unsigned ep_a, Prof &pr, RingPos &rp, uint32_t ring_s, int slot_bytes,
                                               uint64_t *myfull, uint64_t *empty) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float4 *sq = reinterpret_cast<float4 *>(scratch);  // [KVMUL][32]
    float4 *sk = sq + KVMUL * 32;                      // [32]
    float4 *sv = sk + 32;                              // [32]
    float *sbase = reinterpret_cast<float *>(sv + 32); // behind q / k / v: scores, then the merge of the two groups
    static_assert((KVMUL * 32 + 64) * 16 + (2 * MEGA_GW * 32 + 16 + 8 * HEAD_DIM) * 4 <= MEGA_SCRATCH, "attention scratch");
    static_assert(KVMUL + 2 <= MEGA_NCW, "one warp per gathered row");
    const int n = pos + 1;
    const int per = (n + nsplit - 1) / nsplit;
    const int t0 = split * per;
    int t1 = t0 + per;
    if (t1 > n) t1 = n;
    const bool owner = pos >= t0 && pos < t1; // this split attends to (and stores) the new position
    float *kc_l = a.kc + (size_t)layer * a.seq_len * a.KV_l;
    float *vc_l = a.vc + (size_t)layer * a.seq_len * a.KV_l;
    if (warp < KVMUL + 2 && (warp < KVMUL || owner)) {
        const bool isq = warp < KVMUL, isk = warp == KVMUL;
        // static operands first: their loaded latency overlaps the poll
        float4 wv = make_float4(0.f, 0.f, 0.f, 0.f), cs01 = wv, cs23 = wv;
        if (isq || isk) {
            wv = __ldg(reinterpret_cast<const float4 *>((isq ? a.q_ln : a.k_ln) + (size_t)layer * HEAD_DIM) + lane);
            const float4 *cs = reinterpret_cast<const float4 *>(a.rope + (size_t)pos * HEAD_DIM) + (lane & 15) * 2;
            cs01 = __ldg(cs);
            cs23 = __ldg(cs + 1);
        }
        const int row0 = isq ? (kvh * KVMUL + warp) * HEAD_DIM : (isk ? a.AH_l : a.AH_l + a.KV_l) + kvh * HEAD_DIM;
        const float4 v = ll_poll4(a, a.zq + row0 + lane * 4, ep_q, 9);
        if (isq) {
            sq[warp * 32 + lane] = qk_norm_rope_pre(v, wv, cs01, cs23, lane);
        } else if (isk) {
            const float4 r = qk_norm_rope_pre(v, wv, cs01, cs23, lane);
            sk[lane] = r;
            reinterpret_cast<float4 *>(kc_l + (size_t)pos * a.KV_l + (size_t)kvh * HEAD_DIM)[lane] = r;
        } else {
            sv[lane] = v;
            reinterpret_cast<float4 *>(vc_l + (size_t)pos * a.KV_l + (size_t)kvh * HEAD_DIM)[lane] = v;
        }
    }
    csync();
    prof_mark(pr, 35); // q / k normalised + rotated
    const float scale = __fdiv_rn(1.0f, sqrtf((float)HEAD_DIM));
    float4 A = make_float4(0.f, 0.f, 0.f, 0.f);
    float M = -INFINITY, L = 0.0f;
    {
        // The cache rows t0 .. t1 of this kv head arrive through the weight ring: stages of MEGA_KV_ROWS = 32 positions (K tile, then
        // V tile, 16 KB each, [position][128] f32), issued by the producers behind the QKV weights; stages alternate between the two
        // consumer groups like weight stages.  Inside a group, warp w works for query head w % KVMUL on the dims of part w / KVMUL
        // (PARTS = 8 / KVMUL parts of DPP dims):
        //   scores : LANE = cached position.  Each lane walks its K row in 16-byte chunks, starting `lane` chunks in (the rows are
        //            512 B apart, so the same chunk index in every lane would be a 32-way bank conflict; skewed, a quarter warp
        //            touches 8 distinct bank groups, and the matching q chunks are consecutive addresses); the PARTS partial sums
        //            of a head are exchanged through shared memory;
        //   softmax: ONE update per 32 positions -- a warp maximum, one exp per lane, a warp sum (a loop with lane = dims redoes
        //            the whole online update, 2 exps, in all 32 lanes for every single position);
        //   P V    : lane = dims; the weight of position j comes from lane j by shuffle.
        // Row `pos` itself is not in the cache yet when its tile is fetched: that lane / iteration reads sk / sv instead.
        constexpr int PARTS = MEGA_GW / KVMUL, DPP = HEAD_DIM / PARTS, CPP = DPP / 4; // dims / 16-byte chunks per part
        constexpr int VPL = DPP >= 32 ? DPP / 32 : 1;                                  // output dims per lane (KVMUL 1: lanes >= DPP idle)
        static_assert(MEGA_GW % KVMUL == 0 && (CPP & (CPP - 1)) == 0, "head / part split");
        const int grp = warp / MEGA_GW, wl = warp % MEGA_GW;
        const int head = wl % KVMUL, part = wl / KVMUL;
        float *sS = sbase + grp * (MEGA_GW * 32);                                       // [grp][part][head][32] partial scores
        const uint32_t sq_s = smem_u32(sq) + head * 512, sk_s = smem_u32(sk), sv_s = smem_u32(sv);
        float m = -INFINITY, l = 0.0f;
        float acc[VPL];
#pragma unroll
        for (int j = 0; j < VPL; j++) acc[j] = 0.0f;
        const int nst = (t1 - t0 + MEGA_KV_ROWS - 1) / MEGA_KV_ROWS;
        for (int st = 0; st < nst; st++) {
            if ((st & 1) == grp) {
                const int slot = rp.it % MEGA_NSTAGE;
                mbar_wait(&myfull[slot], (rp.fullp >> slot) & 1, a.status);
                rp.fullp ^= 1u << slot;
                const uint32_t kt = ring_s + slot * slot_bytes, vt = kt + MEGA_KV_ROWS * HEAD_DIM * 4;
                const int tb = t0 + st * MEGA_KV_ROWS, t = tb + lane; // first position of the stage, this lane's position
                const uint32_t krow = (t == pos ? sk_s : kt + lane * (HEAD_DIM * 4)) + part * (DPP * 4);
                const uint32_t qrow = sq_s + part * (DPP * 4);
                // four chunks per round: eight 128-bit loads in flight, four independent partial sums
                float s4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                for (int i0 = 0; i0 < CPP; i0 += 4) {
                    int4 ki[4], qi[4];
                    uint32_t cc[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) cc[u] = ((i0 + u + lane) & (CPP - 1)) * 16;
                    // one asm statement: left to itself the compiler re-serialises the round into load-load-4 FMAs per chunk (registers),
                    // which exposes a shared-memory latency per chunk
                    asm volatile(
                        "ld.shared.v4.b32 {%0,%1,%2,%3}, [%32];\n\tld.shared.v4.b32 {%4,%5,%6,%7}, [%33];\n\t"
                        "ld.shared.v4.b32 {%8,%9,%10,%11}, [%34];\n\tld.shared.v4.b32 {%12,%13,%14,%15}, [%35];\n\t"
                        "ld.shared.v4.b32 {%16,%17,%18,%19}, [%36];\n\tld.shared.v4.b32 {%20,%21,%22,%23}, [%37];\n\t"
                        "ld.shared.v4.b32 {%24,%25,%26,%27}, [%38];\n\tld.shared.v4.b32 {%28,%29,%30,%31}, [%39];"
                        : "=r"(ki[0].x), "=r"(ki[0].y), "=r"(ki[0].z), "=r"(ki[0].w), "=r"(ki[1].x), "=r"(ki[1].y), "=r"(ki[1].z), "=r"(ki[1].w),
                          "=r"(ki[2].x), "=r"(ki[2].y), "=r"(ki[2].z), "=r"(ki[2].w), "=r"(ki[3].x), "=r"(ki[3].y), "=r"(ki[3].z), "=r"(ki[3].w),
                          "=r"(qi[0].x), "=r"(qi[0].y), "=r"(qi[0].z), "=r"(qi[0].w), "=r"(qi[1].x), "=r"(qi[1].y), "=r"(qi[1].z), "=r"(qi[1].w),
                          "=r"(qi[2].x), "=r"(qi[2].y), "=r"(qi[2].z), "=r"(qi[2].w), "=r"(qi[3].x), "=r"(qi[3].y), "=r"(qi[3].z), "=r"(qi[3].w)
                        : "r"(krow + cc[0]), "r"(krow + cc[1]), "r"(krow + cc[2]), "r"(krow + cc[3]), "r"(qrow + cc[0]), "r"(qrow + cc[1]),
                          "r"(qrow + cc[2]), "r"(qrow + cc[3]));
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        s4[u] = fmaf(__int_as_float(qi[u].x), __int_as_float(ki[u].x), s4[u]);
                        s4[u] = fmaf(__int_as_float(qi[u].y), __int_as_float(ki[u].y), s4[u]);
                        s4[u] = fmaf(__int_as_float(qi[u].z), __int_as_float(ki[u].z), s4[u]);
                        s4[u] = fmaf(__int_as_float(qi[u].w), __int_as_float(ki[u].w), s4[u]);
                    }
                }
                float s = (s4[0] + s4[1]) + (s4[2] + s4[3]);
                if (PARTS > 1) { // the parts of a head add their partial sums (same order in every part: identical scores)
                    sS[(part * KVMUL + head) * 32 + lane] = s;
                    gsync(grp);
                    s = 0.0f;
#pragma unroll
                    for (int pp = 0; pp < PARTS; pp++) s += sS[(pp * KVMUL + head) * 32 + lane];
                    gsync(grp); // sS is rewritten in this group's next stage
                }
                s = t < t1 ? __fmul_rn(s, scale) : -INFINITY;
                const float mn = fmaxf(m, warp_max(s));
                const float corr = expf(m - mn), pj = expf(s - mn); // exp(-inf) = 0: first stage / positions past the end
                l = l * corr + warp_sum(pj);
                m = mn;
#pragma unroll
                for (int j = 0; j < VPL; j++) acc[j] *= corr;
                // all 32 rows of the stage, four per round (loads and shuffles of a round in flight together): rows past the end carry
                // weight 0 (their scores were -inf) and finite values (cache rows are zero-initialised, tiles past the cache zero-filled)
                const uint32_t vcol = (part * DPP + (DPP >= 32 ? lane * VPL : (lane & (DPP - 1)))) * 4;
                const int jpos = pos - tb; // row of the stage that holds `pos` (taken from sv), if any
#pragma unroll 2
                for (int j0 = 0; j0 < MEGA_KV_ROWS; j0 += 4) {
                    float vv[4][VPL], w[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const uint32_t va = (j0 + u == jpos ? sv_s : vt + (j0 + u) * (HEAD_DIM * 4)) + vcol;
                        if (VPL == 4) {
                            const int4 v = lds128(va);
                            vv[u][0] = __int_as_float(v.x);
                            vv[u][1 % VPL] = __int_as_float(v.y);
                            vv[u][2 % VPL] = __int_as_float(v.z);
                            vv[u][3 % VPL] = __int_as_float(v.w);
                        } else if (VPL == 2) {
                            asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(vv[u][0]), "=f"(vv[u][1 % VPL]) : "r"(va));
                        } else {
                            vv[u][0] = lds_f32(va);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) w[u] = __shfl_sync(0xffffffffu, pj, j0 + u);
#pragma unroll
                    for (int u = 0; u < 4; u++)
#pragma unroll
                        for (int j = 0; j < VPL; j++) acc[j] = fmaf(w[u], vv[u][j], acc[j]);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[slot]);
            }
            rp.it++;
        }
        prof_mark(pr, 36); // position loop done
        // merge the two groups (each holds the stages it owned), head by head: group 1 hands over, group 0 combines and lays the head
        // out as [128] floats for the warps that publish it
        float *xm = sbase, *xl = sbase + 2 * MEGA_GW * 32;                      // group 1's m[8] (score area, free now) and l[8]
        float *xa = xl + 16;                                                   // group 1's accumulators [8 warps][DPP], then the final [KVMUL][128]
        csync(); // every warp is done with sS
        if (grp == 1) {
            if (lane == 0) {
                xm[wl] = m;
                xl[wl] = l;
            }
            if (DPP >= 32 || lane < DPP) {
#pragma unroll
                for (int j = 0; j < VPL; j++) xa[wl * DPP + (DPP >= 32 ? lane * VPL : lane) + j] = acc[j];
            }
        }
        csync();
        float mt = m, lt = l;
        if (grp == 0) {
            const float m1 = xm[wl], l1 = xl[wl];
            mt = fmaxf(m, m1);
            const float c0 = m == -INFINITY ? 0.0f : expf(m - mt), c1 = m1 == -INFINITY ? 0.0f : expf(m1 - mt);
            lt = l * c0 + l1 * c1;
            if (DPP >= 32 || lane < DPP) {
#pragma unroll
                for (int j = 0; j < VPL; j++) {
                    const int d = (DPP >= 32 ? lane * VPL : lane) + j;
                    acc[j] = acc[j] * c0 + xa[wl * DPP + d] * c1;
                }
            }
        }
        csync(); // group 1's hand-over has been read: xa becomes the [KVMUL][128] output layout
        float *xo = xa, *xs_m = sbase + 16, *xs_l = sbase + 24; // (free part of the score area)
        if (grp == 0) {
            if (DPP >= 32 || lane < DPP) {
#pragma unroll
                for (int j = 0; j < VPL; j++) xo[head * HEAD_DIM + part * DPP + (DPP >= 32 ? lane * VPL : lane) + j] = acc[j];
            }
            if (part == 0 && lane == 0) {
                xs_m[head] = mt;
                xs_l[head] = lt;
            }
        }
        csync();
        if (warp < KVMUL) {
            A = reinterpret_cast<const float4 *>(xo + warp * HEAD_DIM)[lane];
            M = xs_m[warp];
            L = xs_l[warp];
        }
    }
    if (nsplit == 1) { // the only split of its kv head: A / L is the attention output
        if (warp < KVMUL) publish_head<GS>(a, kvh * KVMUL + warp, lane, A, L, ep_a);
        return;
    }
    if (warp < KVMUL) {
        float *dst = a.attn_part + ((size_t)(kvh * KVMUL + warp) * MEGA_MAX_SPLITS + split) * ATTN_PART_STRIDE;
        reinterpret_cast<float4 *>(dst)[lane] = A;
        if (lane == 0) {
            dst[HEAD_DIM] = M;
            dst[HEAD_DIM + 1] = L;
        }
    }
    unsigned *flag = reinterpret_cast<unsigned *>(sbase); // group 1's hand-over, consumed above
    csync();
    if (tid == 0) {
        __threadfence();
        unsigned *cnt = a.att_cnt + (size_t)layer * a.n_kv_l + kvh;
        const unsigned old = atomicAdd(cnt, 1u);
        const bool is_last = old == (unsigned)nsplit - 1;
        if (is_last) *cnt = 0; // every split of this (layer, kv head) has arrived; next use is the next launch
        __threadfence();
        *flag = is_last ? 1u : 0u;
    }
    csync();
    prof_mark(pr, 37); // split partial stored, arrival counted
    if (*flag != 0 && warp < KVMUL) {
        // Lane s first fetches the statistics of split s (one memory round trip for all splits), then the partial
        // accumulators are pulled four splits at a time.
        const int head = kvh * KVMUL + warp;
        const float *pb = a.attn_part + (size_t)head * MEGA_MAX_SPLITS * ATTN_PART_STRIDE;
        const float ms = lane < nsplit ? ldcg_f(pb + lane * ATTN_PART_STRIDE + HEAD_DIM) : -INFINITY;
        const float ls = lane < nsplit ? ldcg_f(pb + lane * ATTN_PART_STRIDE + HEAD_DIM + 1) : 0.0f;
        const float Mx = warp_max(ms);
        const float cs = lane < nsplit ? expf(ms - Mx) : 0.0f;
        const float Ls = warp_sum(ls * cs);
        float4 As = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
        for (int s0 = 0; s0 < nsplit; s0 += 4) {
            float4 pv[4];
#pragma unroll
            for (int j = 0; j < 4; j++)
                pv[j] = (s0 + j < nsplit) ? ldcg_f4(pb + (s0 + j) * ATTN_PART_STRIDE + lane * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const float c = __shfl_sync(0xffffffffu, cs, (s0 + j) & 31);
                As.x += pv[j].x * c;
                As.y += pv[j].y * c;
                As.z += pv[j].z * c;
                As.w += pv[j].w * c;
            }
        }
        publish_head<GS>(a, head, lane, As, Ls, ep_a);
    }
}

// ------------------------------------------------------------------------------------------
// grid barrier (once per token, before the greedy argmax; + cross-GPU arrival under TP)
// ------------------------------------------------------------------------------------------
struct BarState {
    unsigned long long target;  // next value the local counter must reach
    unsigned long long xtarget; // next value this rank's cross-GPU counter must reach
};

// Local: every CTA adds 1 to this GPU's counter and waits for gridDim.x arrivals.
// Cross (tensor parallel): every CTA of every rank adds 1 to the counter of EVERY rank (remote reductions over NVLink)
// and waits for tp * gridDim.x arrivals on its own -- one system-scope fence and one NVLink one-way trip, no second hop
// through a leader CTA.
__device__ __noinline__ void grid_barrier(const MegaArgs &a, BarState &bs, bool cross, Prof &pr) {
    csync();
    prof_mark(pr, 40); // all consumer warps of this CTA done
    const bool x = cross && a.tp_size > 1;
    if (threadIdx.x == 0) {
        long long t0 = clock64();
        volatile int *st = a.status;
        unsigned spins = 0;
        if (x) {
            __threadfence_system(); // this CTA's stores (cumulative over bar.sync), incl. the P2P ones, before the arrivals
            for (int r = 0; r < a.tp_size; r++)
                asm volatile("red.relaxed.sys.global.add.u64 [%0], %1;" ::"l"(a.xbar[r]), "l"(1ULL) : "memory");
            while (true) {
                unsigned long long v;
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(a.xbar[a.tp_rank]) : "memory");
                if (v >= bs.xtarget) break;
                if ((++spins & 1023u) == 0) {
                    if (*st) break;
                    if (clock64() - t0 > 8000000000LL) {
                        atomicExch(a.status, 3);
                        break;
                    }
                }
            }
        } else {
            // one release-reduction (no return value to wait for); bar.sync above makes the other threads'
            // stores cumulative with it
            asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(a.bar), "l"(1ULL) : "memory");
            while (true) {
                unsigned long long v;
                asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(a.bar) : "memory");
                if (v >= bs.target) break;
                if ((++spins & 1023u) == 0) {
                    if (*st) break;
                    if (clock64() - t0 > 4000000000LL) {
                        atomicExch(a.status, 1);
                        break;
                    }
                }
            }
        }
    }
    if (x) bs.xtarget += (unsigned long long)a.tp_size * gridDim.x;
    else bs.target += gridDim.x;
    prof_mark(pr, 41); // all CTAs arrived (seen by thread 0)
    csync();
}

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
struct PhaseGeom {
    const uint8_t *seg; // this CTA's segment of the phase stream
    int start, count;   // units owned by this CTA
};
// per-CTA constants computed once (integer divisions are ~40 instructions each on the GPU)
struct MegaShared {
    int start[5], count[5];
    long long seg_off[5], seg_len[5];
    unsigned long long *part[2][MEGA_MAX_TP];
    float *logits[MEGA_MAX_TP];
    unsigned long long *best[MEGA_MAX_TP];
};
__device__ __forceinline__ PhaseGeom phase_geom(const MegaArgs &a, const MegaShared &sh, int ph, int layer) {
    PhaseGeom pg;
    pg.start = sh.start[ph];
    pg.count = sh.count[ph];
    pg.seg = a.g[ph].base + (long long)layer * a.g[ph].layer_stride + sh.seg_off[ph];
    return pg;
}

template <int GS, int KVMUL>
__global__ void __launch_bounds__(MEGA_THREADS, 1) k_mega_decode(const __grid_constant__ MegaArgs a) {
    extern __shared__ __align__(1024) uint8_t mega_smem[];
    uint8_t *smem = mega_smem;
    // layout: [ring: NSTAGE x slot][scratch][barriers + per-CTA constants][residual stream]
    const int slot_bytes = MEGA_GW * (MEGA_MAX_KT + 4 * (MEGA_MAX_KT / GS));
    uint8_t *ring = smem;
    uint8_t *scratch = smem + MEGA_NSTAGE * slot_bytes;
    uint8_t *sxq = scratch;                                          // up to 16384 B
    float *sxs = reinterpret_cast<float *>(scratch + 16384);         // up to 512 groups
    float *sred = reinterpret_cast<float *>(scratch + 16384 + 2048); // 16 floats (+ argmax scratch at +32)
    // full barriers are per (consumer group, slot): a waiter can only tell adjacent mbarrier phases
    // apart, and with ownership alternating between the groups a group would otherwise skip the
    // other group's use of a slot and mistake the phase before it for its own.
    uint64_t *full = reinterpret_cast<uint64_t *>(scratch + MEGA_SCRATCH); // [MEGA_GROUPS][MEGA_NSTAGE]
    uint64_t *empty = full + MEGA_GROUPS * MEGA_NSTAGE;                    // [MEGA_NSTAGE]
    MegaShared &sh = *reinterpret_cast<MegaShared *>(scratch + MEGA_SCRATCH + 192);
    static_assert(192 + sizeof(MegaShared) <= 1024, "MegaShared outgrew its slot");
    float *sx = reinterpret_cast<float *>(scratch + MEGA_SCRATCH + 1024); // residual stream, MEGA_MAX_KT floats
    volatile unsigned *issued = reinterpret_cast<volatile unsigned *>(scratch + MEGA_SCRATCH + 128); // [MEGA_NSTAGE] uses issued per slot
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
        for (int s = 0; s < MEGA_NSTAGE; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&full[MEGA_NSTAGE + s], 1);
            mbar_init(&empty[s], MEGA_GW);
            issued[s] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll 1
        for (int ph = 0; ph < 5; ph++) {
            int st, cn;
            cta_share(a.g[ph].units, gridDim.x, blockIdx.x, st, cn);
            const long long per_unit = (long long)(ph == PH_GU ? 2 : 1) * a.g[ph].n_kt * a.g[ph].tile_bytes;
            sh.start[ph] = st;
            sh.count[ph] = cn;
            sh.seg_off[ph] = st * per_unit;
            sh.seg_len[ph] = cn * per_unit;
        }
    }
    if (tid < MEGA_MAX_TP) {
        sh.part[0][tid] = a.part[0][tid];
        sh.part[1][tid] = a.part[1][tid];
        sh.logits[tid] = a.logits[tid];
        sh.best[tid] = a.best[tid];
    }
    __syncthreads();

    const int L0 = a.layer0, L1 = a.layer1;

    if (warp >= MEGA_NCW) {
        // =============================== PRODUCERS ===============================
        // One producer thread per consumer group: the serial wait -> expect_tx -> bulk-copy loop of a single
        // thread (~0.6 us per stage) capped how fast the ring could refill; two threads issue independently,
        // each feeding the stages its group owns.
        if (lane != 0) return;
        const int pw = warp - MEGA_NCW;
        uint64_t policy;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
        unsigned it = 0;
        Prof pr; // producer 0 logs every stage it issues (tag 64 + slot) into a second row per CTA
        pr.row = (a.prof && pw == 0) ? a.prof + (size_t)(gridDim.x + blockIdx.x) * MEGA_PROF_EVENTS : nullptr;
        pr.ev = 0;
        auto push = [&](const uint8_t *src, int nr, int tile_bytes, int owner) {
            if (owner != pw) { // the other producer's stage
                it++;
                return;
            }
            const int slot = it % MEGA_NSTAGE;
            const uint32_t bytes = (uint32_t)nr * tile_bytes;
            // The two producers share the slots.  A waiter can only tell adjacent mbarrier phases apart, so
            // before waiting for "use n-1 of this slot released" make sure use n-1 has been ISSUED (by the
            // other producer) -- otherwise an early arrival would mistake use n-3's release for it.
            {
                const unsigned use = it / MEGA_NSTAGE;
                long long t0 = clock64();
                while (issued[slot] != use) {
                    if (clock64() - t0 > 4000000000LL) { atomicExch(a.status, 4); break; }
                }
            }
            mbar_wait(&empty[slot], ((it / MEGA_NSTAGE) & 1) ^ 1, a.status);
            uint64_t *fb = &full[owner * MEGA_NSTAGE + slot];
            mbar_expect_tx(fb, bytes);
            bulk_g2s(ring + (size_t)slot * slot_bytes, src, bytes, fb, policy);
            __threadfence_block();
            issued[slot] = it / MEGA_NSTAGE + 1;
            prof_mark(pr, 64 + slot);
            it++;
        };
        // K/V cache tiles of this CTA's attention item (kv head, split) for `layer`: same slots, same handshake as weight stages
        const int ppos = a.tokpos[1];
        const int pns = mega_nsplit(ppos, a.n_kv_l, gridDim.x);
        const bool has_item = (int)blockIdx.x < a.n_kv_l * pns;
        const int pkvh = blockIdx.x % a.n_kv_l, psplit = blockIdx.x / a.n_kv_l;
        const int pper = (ppos + 1 + pns - 1) / pns;
        const int pt0 = psplit * pper, pt1 = pt0 + pper < ppos + 1 ? pt0 + pper : ppos + 1;
        auto kvpush = [&](int layer) {
            if (!has_item) return;
            for (int t = pt0, si = 0; t < pt1; t += MEGA_KV_ROWS, si++) {
                const int owner = si & 1;
                if (owner != pw) {
                    it++;
                    continue;
                }
                const int slot = it % MEGA_NSTAGE;
                {
                    const unsigned use = it / MEGA_NSTAGE;
                    long long tw = clock64();
                    while (issued[slot] != use) {
                        if (clock64() - tw > 4000000000LL) { atomicExch(a.status, 4); break; }
                    }
                }
                mbar_wait(&empty[slot], ((it / MEGA_NSTAGE) & 1) ^ 1, a.status);
                uint64_t *fb = &full[owner * MEGA_NSTAGE + slot];
                uint8_t *dst = ring + (size_t)slot * slot_bytes;
                mbar_expect_tx(fb, 2 * MEGA_KV_ROWS * HEAD_DIM * 4);
                tma_load_2d(dst, &a.map_k, pkvh * HEAD_DIM, layer * a.seq_len + t, fb);
                tma_load_2d(dst + MEGA_KV_ROWS * HEAD_DIM * 4, &a.map_v, pkvh * HEAD_DIM, layer * a.seq_len + t, fb);
                __threadfence_block();
                issued[slot] = it / MEGA_NSTAGE + 1;
                prof_mark(pr, 64 + slot);
                it++;
            }
        };
        auto plain = [&](int ph, int layer) {
            const MegaGemv &g = a.g[ph];
            PhaseGeom pg = phase_geom(a, sh, ph, layer);
            const uint8_t *src = pg.seg;
            for (int b0 = 0; b0 < pg.count; b0 += MEGA_BATCH) {
                int nb = pg.count - b0 < MEGA_BATCH ? pg.count - b0 : MEGA_BATCH;
                for (int kt = 0; kt < g.n_kt; kt++)
                    for (int s = 0, si = 0; s < nb; s += MEGA_GW, si++) {
                        int nr = nb - s < MEGA_GW ? nb - s : MEGA_GW;
                        push(src, nr, g.tile_bytes, si & 1);
                        src += (size_t)nr * g.tile_bytes;
                    }
            }
        };
        auto pairs = [&](int layer) {
            const MegaGemv &g = a.g[PH_GU];
            PhaseGeom pg = phase_geom(a, sh, PH_GU, layer);
            const uint8_t *src = pg.seg;
            for (int p0 = 0, bi = 0; p0 < pg.count; p0 += MEGA_GW, bi++) {
                int np = pg.count - p0 < MEGA_GW ? pg.count - p0 : MEGA_GW;
                for (int half = 0; half < 2; half++) {
                    push(src, np, g.tile_bytes, bi & 1);
                    src += (size_t)np * g.tile_bytes;
                }
            }
        };
        for (int l = L0; l < L1; l++) {
            plain(PH_QKV, l);
            kvpush(l);
            plain(PH_O, l);
            pairs(l);
            plain(PH_DN, l);
        }
        if (a.run_head) plain(PH_HEAD, 0);
        if (pr.row) pr.row[MEGA_PROF_EVENTS - 1] = (unsigned long long)pr.ev;
        return;
    }

    // =============================== CONSUMERS ===============================
    // The forward pass is walked as a flat sequence of steps (5 per layer + the head) through ONE
    // copy of each code path: the per-token instruction footprint has to stay inside the
    // instruction cache -- an earlier version that inlined a GEMV loop per phase was 340 KB of SASS
    // and spent more time fetching instructions (through the same L2 the weights stream through)
    // than computing.
    unsigned it = 0;
    BarState bs;
    bs.target = a.bar_base + gridDim.x;
    bs.xtarget = a.xbar_base + (unsigned long long)a.tp_size * gridDim.x;
    const int pos = a.tokpos[1];
    const int grp = warp / MEGA_GW, wl = warp % MEGA_GW; // consumer group and warp-in-group (= row tile in a stage)
    Prof pr;
    pr.row = (a.prof && (tid == 0 || tid == MEGA_GW * 32)) ? a.prof + (size_t)((tid ? 2 * gridDim.x : 0) + blockIdx.x) * MEGA_PROF_EVENTS : nullptr; // + first lane of group 1
    pr.ev = 0;
    unsigned fullp = 0; // bit s: parity of this group's next use of slot s
    uint64_t *myfull = full + grp * MEGA_NSTAGE;
    XRegs<GS> xr;
    prof_mark(pr, 0);
    long long best = (long long)0x8000000000000000LL;
    const int n_layer_steps = 5 * (L1 - L0);
    const int n_steps = n_layer_steps + (a.run_head ? 1 : 0);
    const int nsplit = mega_nsplit(pos, a.n_kv_l, gridDim.x);

    for (int step = 0; step < n_steps; step++) {
        const bool head = step >= n_layer_steps;
        const int l = head ? 0 : L0 + step / 5;
        const int kind = head ? 5 : step % 5; // 0 qkv, 1 attention, 2 o_proj, 3 gate/up, 4 down, 5 lm_head
        // epoch of step (l, kind): everything a step publishes carries it (each zone is written by one step kind, or by
        // steps that are never in flight together); the head step takes the slot after the last layer
        const unsigned ep_step = ll_epoch(a.ll_base, head ? (unsigned)(MEGA_EDGES * (L1 - L0)) : (unsigned)(MEGA_EDGES * (l - L0) + kind));
        const unsigned ep_prev = ll_epoch(a.ll_base, (unsigned)(MEGA_EDGES * (l - L0) + kind - 1)); // of the preceding step of this layer
        int ph = PH_QKV;
        // ------------------------------ prologue ------------------------------
        if (kind == 0 || kind == 3 || kind == 5) {
            // RMSNorm + quantize of the residual stream (qwen3.rs:134-136, 159-161, 72-75)
            const float *w = kind == 0 ? a.rms_att + (size_t)l * a.dim : kind == 3 ? a.rms_ffn + (size_t)l * a.dim : a.rms_final;
            const bool emb = kind == 0 && l == L0 && a.from_embed;
            const bool pending = kind == 3 || (kind == 0 ? l > L0 : L1 > L0); // a row-parallel GEMV (o_proj / down) has just run
            ph = kind == 0 ? PH_QKV : kind == 3 ? PH_GU : PH_HEAD;
            // rows being consumed: o_proj of this layer (kind 3) or down of the previous / last layer
            const unsigned ep_rows = kind == 3 ? ep_prev : ll_epoch(a.ll_base, (unsigned)(MEGA_EDGES * ((kind == 0 ? l - 1 : L1 - 1) - L0) + 4));
            prologue_norm<GS>(a, w, emb ? 0 : (pending ? 2 : 1), pending ? a.zr[kind == 3 ? 0 : 1] : nullptr, ep_rows, sxq, sxs, sred, sx,
                              a.g[ph].KT, a.g[ph].G, pr);
        } else if (kind == 1) {
            // QK-norm + RoPE + attention (layers.rs:339-343) + quantize (qwen3.rs:152) on the CTAs that own a (kv head, split) item
            if ((int)blockIdx.x < a.n_kv_l * nsplit) {
                RingPos rp{it, fullp};
                attention_item<GS, KVMUL>(a, l, pos, blockIdx.x % a.n_kv_l, blockIdx.x / a.n_kv_l, nsplit, scratch, ep_prev, ep_step, pr, rp,
                                          smem_u32(ring), slot_bytes, myfull, empty);
                it = rp.it;
                fullp = rp.fullp;
            }
        } else if (kind == 2) {
            prologue_attn_poll<GS>(a, ep_prev, sxq, sxs);
            ph = PH_O;
        } else {
            prologue_quant_ll<GS>(a, a.zh, ep_prev, a.H_l, sxq, sxs, a.g[PH_DN].KT, a.g[PH_DN].G); // quantize(hb), layers.rs:478
            ph = PH_DN;
        }
        prof_mark(pr, 1 + 3 * kind);
        // ------------------------------ GEMV ------------------------------
        if (kind != 1) {
            const MegaGemv &g = a.g[ph];
            const int start = sh.start[ph], count = sh.count[ph];
            const bool full_blocks = (g.G & 31) == 0;
            const uint32_t ring_s = smem_u32(ring);
            if (kind == 3) {
                // gate/up + SwiGLU (layers.rs:468-475): blocks of 8 pairs, a gate stage then an up stage
                const unsigned ep_h = ep_step;
                load_x<GS>(xr, sxq, sxs, 0, g.KT, g.G, lane);
                for (int p0 = 0, bi = 0; p0 < count; p0 += MEGA_GW, bi++) {
                    const int np = count - p0 < MEGA_GW ? count - p0 : MEGA_GW;
                    if ((bi & 1) != grp) { // blocks alternate between the consumer groups
                        it += 2;
                        continue;
                    }
                    float gate = 0.0f, up = 0.0f;
                    for (int half = 0; half < 2; half++) {
                        const int slot = it % MEGA_NSTAGE;
                        mbar_wait(&myfull[slot], (fullp >> slot) & 1, a.status);
                        fullp ^= 1u << slot;
                        prof_mark(pr, 48 + slot);
                        {   // every warp runs the dot (warp-convergent shuffles); a warp without a row reads stale smem and drops the value
                            const uint32_t tile = ring_s + slot * slot_bytes + wl * g.tile_bytes;
                            float v = full_blocks ? tile_dot<GS, true>(tile, xr, g.KT, g.G, lane) : tile_dot<GS, false>(tile, xr, g.KT, g.G, lane);
                            gate = half == 0 ? v : gate;
                            up = half == 0 ? up : v;
                        }
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty[slot]);
                        it++;
                    }
                    if (wl < np && lane == 0) {
                        float sw = __fmul_rn(gate, __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-gate))));
                        ll_store(a.zh + start + p0 + wl, __fmul_rn(sw, up), ep_h);
                    }
                }
            } else {
                // row phases: batches of 32 rows x n_kt K tiles x up to 4 stages of 8 rows
                const unsigned ep_out = ep_step;
                for (int b0 = 0; b0 < count; b0 += MEGA_BATCH) {
                    const int nb = count - b0 < MEGA_BATCH ? count - b0 : MEGA_BATCH;
                    float acc0 = 0.f, acc1 = 0.f; // this warp's rows in its (up to) two stages of the batch
                    for (int kt = 0; kt < g.n_kt; kt++) {
                        load_x<GS>(xr, sxq, sxs, kt, g.KT, g.G, lane);
                        prof_mark(pr, 58);
                        for (int sidx = 0; MEGA_GW * sidx < nb; sidx++) {
                            if ((sidx & 1) == grp) { // stages alternate between the two consumer groups
                                const int slot = it % MEGA_NSTAGE;
                                mbar_wait(&myfull[slot], (fullp >> slot) & 1, a.status);
                                fullp ^= 1u << slot;
                                prof_mark(pr, 48 + slot);
                                {
                                    const uint32_t tile = ring_s + slot * slot_bytes + wl * g.tile_bytes;
                                    float v = full_blocks ? tile_dot<GS, true>(tile, xr, g.KT, g.G, lane) : tile_dot<GS, false>(tile, xr, g.KT, g.G, lane);
                                    v = (MEGA_GW * sidx + wl < nb) ? v : 0.0f; // warp without a row: stale smem, value dropped
                                    acc0 += sidx < 2 ? v : 0.0f;
                                    acc1 += sidx < 2 ? 0.0f : v;
                                    prof_mark(pr, 59);
                                }
                                __syncwarp();
                                if (lane == 0) mbar_arrive(&empty[slot]);
                            }
                            it++;
                        }
                    }
                    // epilogue: lane 0 of the owning warp, rows (grp) and (grp + 2) of the batch's stages
                    if (lane == 0) {
                        for (int j = 0; j < 2; j++) {
                            const int sidx = grp + 2 * j;
                            if (MEGA_GW * sidx + wl >= nb) break;
                            const int r = start + b0 + MEGA_GW * sidx + wl;
                            const float v = j == 0 ? acc0 : acc1;
                            if (kind == 0) { // layers.rs:334-336: q | k | v rows, picked up by the attention CTAs
                                ll_store(a.zq + r, v, ep_out);
                            } else if (kind == 2 || kind == 4) {
                                if (a.tp_size == 1) { // the row is complete: straight into the zone every prologue polls
                                    ll_store(a.zr[kind == 2 ? 0 : 1] + r, v, ep_out);
                                } else { // row-parallel partial -> every rank's landing zone (peer stores over NVLink)
                                    unsigned long long *const *dst = sh.part[kind == 2 ? 0 : 1];
#pragma unroll 1
                                    for (int p = 0; p < a.tp_size; p++) ll_store(dst[p] + (size_t)a.tp_rank * a.dim + r, v, ep_out);
                                }
                            } else { // lm_head (qwen3.rs:76) + greedy argmax candidate (sampler.rs:57-59)
                                const int row = a.vocab_row0 + r;
                                sh.logits[a.tp_rank][row] = v;
                                if (a.gather_logits) { // bit p: rank p wants the full-vocabulary logits (peer stores over NVLink)
#pragma unroll 1
                                    for (int p = 0; p < a.tp_size; p++)
                                        if (p != a.tp_rank && ((a.gather_logits >> p) & 1)) sh.logits[p][row] = v;
                                }
                                long long key = ((long long)total_key(v) << 32) | (unsigned)row;
                                best = key > best ? key : best;
                            }
                        }
                    }
                }
                // Tensor parallel all-reduce, two hops regardless of tp: the CTA that computed rows [start, start + count) of
                // this rank's partial also REDUCES those rows -- it polls the tp partial words of each (own word included),
                // adds them in rank order (so every rank computes bit-identical sums) and republishes the row in the local
                // zone every prologue polls.  Each CTA reads tp * count words instead of all CTAs reading tp * dim.
                if ((kind == 2 || kind == 4) && a.tp_size > 1) {
                    const unsigned long long *src = sh.part[kind == 2 ? 0 : 1][a.tp_rank];
                    for (int idx = tid; idx < count; idx += MEGA_CTHREADS) {
                        const int r = start + idx;
                        unsigned long long w[MEGA_MAX_TP];
                        unsigned spins = 0;
                        while (true) {
                            bool ok = true;
#pragma unroll
                            for (int p = 0; p < MEGA_MAX_TP; p++) {
                                if (p < a.tp_size) {
                                    w[p] = ll_load1(src + (size_t)p * a.dim + r);
                                    ok = ok && ll_ok(w[p], ep_out);
                                }
                            }
                            if (ok || ll_give_up(a, spins, 10)) break;
                        }
                        float s = __uint_as_float((unsigned)w[0]);
#pragma unroll
                        for (int p = 1; p < MEGA_MAX_TP; p++)
                            if (p < a.tp_size) s = __fadd_rn(s, __uint_as_float((unsigned)w[p]));
                        ll_store(a.zr[kind == 2 ? 0 : 1] + r, s, ep_out);
                    }
                }
            }
        }
        prof_mark(pr, 2 + 3 * kind);
        if (kind == 5) {
            long long *sbest = reinterpret_cast<long long *>(sred + 32);
            if (lane == 0) sbest[warp] = best;
            csync();
            if (tid == 0) {
                for (int w = 1; w < MEGA_NCW; w++) best = sbest[w] > best ? sbest[w] : best;
#pragma unroll 1
                for (int p = 0; p < a.tp_size; p++) sh.best[p][(size_t)a.tp_rank * gridDim.x + blockIdx.x] = (unsigned long long)best;
            }
        }
        // pull what the next step's first instructions will miss on (static weights, HBM-cold) into L2:
        // the next RMSNorm weight, or the QK-norm weights + this position's RoPE row
        if (kind == 2 || kind == 4) {
            const float *wn = kind == 2 ? a.rms_ffn + (size_t)l * a.dim : (l + 1 < L1 ? a.rms_att + (size_t)(l + 1) * a.dim : a.rms_final);
            if (tid * 32 < a.dim) asm volatile("prefetch.global.L2 [%0];" ::"l"(wn + tid * 32));
        } else if (kind == 0 && tid < 12) {
            const float *wn = tid < 4 ? a.q_ln + (size_t)l * HEAD_DIM + tid * 32 : tid < 8 ? a.k_ln + (size_t)l * HEAD_DIM + (tid - 4) * 32
                                                                                   : a.rope + (size_t)pos * HEAD_DIM + (tid - 8) * 32;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(wn));
        }
        // results carry their own flags: the only thing to wait for is this CTA's own warps (sxq / scratch are about to be rewritten)
        if (kind == 5) grid_barrier(a, bs, true, pr);
        else csync();
        prof_mark(pr, 3 + 3 * kind);
    }

    if (pr.row) pr.row[MEGA_PROF_EVENTS - 1] = (unsigned long long)pr.ev;
    if (a.run_head) {
        if (blockIdx.x == 0 && warp == 0) {
            long long b = (long long)0x8000000000000000LL;
            const int n = a.tp_size * gridDim.x;
            for (int i = lane; i < n; i += 32) {
                long long k = (long long)__ldcg(sh.best[a.tp_rank] + i);
                b = k > b ? k : b;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                long long other = __shfl_xor_sync(0xffffffffu, b, o);
                b = other > b ? other : b;
            }
            if (lane == 0) {
                int tok = (int)(b & 0xffffffffLL);
                a.tokpos[2] = tok;
                if (a.feedback) {
                    a.tokpos[0] = tok;
                    a.tokpos[1] = pos + 1;
                    a.history[a.tokpos[3]] = tok;
                    a.tokpos[3] += 1;
                }
            }
        }
    } else if (blockIdx.x == 0 && L1 > L0) {
        // teacher-forced layer range: materialise x + the last down_proj rows into a.x
        const unsigned ep = ll_epoch(a.ll_base, (unsigned)(MEGA_EDGES * (L1 - 1 - L0) + 4));
        for (int i4 = tid; i4 < (a.dim >> 2); i4 += MEGA_CTHREADS) {
            float4 v = reinterpret_cast<const float4 *>(sx)[i4];
            const float4 d = ll_poll4(a, a.zr[1] + (size_t)i4 * 4, ep, 6);
            v.x = __fadd_rn(v.x, d.x);
            v.y = __fadd_rn(v.y, d.y);
            v.z = __fadd_rn(v.z, d.z);
            v.w = __fadd_rn(v.w, d.w);
            reinterpret_cast<float4 *>(a.x)[i4] = v;
        }
    }
}

} // namespace q3
