// q3_prefill.cuh -- batched (T-token) group-scaled int8 GEMM on the 5th-gen tensor cores.
//
//   out[t, r] = sum_g ( (f32)(sum_{k in g} xq[t,k] * wq[r,k]) * ws[r,g] ) * xs[t,g]        (tensor.rs:41-61, T rows at once)
//
// The int32 accumulator is only meaningful within one quantisation group, so the K loop is cut at
// every group: tcgen05.mma.kind::i8 (A, B int8 from shared memory via TMA, 128B swizzle; D int32
// in TMEM) accumulates GS/32 K-steps into one of four TMEM accumulator buffers, commits, and
// moves on to the next buffer while the epilogue warps drain the previous one
// (tcgen05.ld -> cvt -> (dot*ws)*xs -> f32 add).  Each epilogue thread owns one token row and
// adds its groups in order g = 0..ng-1 with unfused multiplies, i.e. exactly the reference's
// left fold: the GEMM result is bit-identical to `matmul` applied token by token.
//
// Warp roles (608 threads): warps 0..15 = epilogue (TMEM lane quadrant = warp % 4, column quarter = warp / 4: 32 accumulator
// columns per thread keep the register count low enough for 4 epilogue warps per scheduler), warp 16 = TMEM allocator + MMA
// issuer, warp 17 = tile producer (TMA), warp 18 = scale-row producer (TMA).  The single-thread roles sit in the HIGHEST warp ids on purpose: the warp scheduler
// favours the higher warp id among ready warps, and with the roles in warps 0 / 1 the MMA issuer was starved of issue slots
// whenever the four epilogue warps of its scheduler were busy scaling -- the drain arithmetic then did not overlap with the
// tensor pipe at all (measured: time = pipeline-only time + arithmetic time; profiles/r02_gemm_q8_ceilings.txt).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "q3_mega.cuh" // mbarrier helpers

namespace q3 {

constexpr int PF_BM = 128, PF_BN = 128, PF_BK = 128; // tile: tokens x weight rows x K bytes per stage
constexpr int PF_STAGES = 4;
constexpr int PF_NACC = 4;                          // TMEM accumulator buffers (128 columns each), handed over in PAIRS
constexpr int PF_EPI_WARPS = 16;                   // 4 TMEM lane quadrants x 4 column quarters
constexpr int PF_THREADS = (3 + PF_EPI_WARPS) * 32;
constexpr int PF_MMA_WARP = PF_EPI_WARPS, PF_TMA_WARP = PF_EPI_WARPS + 1, PF_SCALE_WARP = PF_EPI_WARPS + 2; // highest warp ids: scheduling priority (see above)
constexpr int PF_COLS = PF_BN / (PF_EPI_WARPS / 4); // accumulator columns per epilogue thread (32)
constexpr int PF_SG = 2;                            // quantisation groups per scale-ring slot: one accumulator pair (even: accumulator pairs never straddle slots)
constexpr int PF_SRING = 8;                         // scale-ring slots: PF_SG x (128 weight scales | 128 token scales) each
constexpr int PF_PATCH_LD = 36;                     // floats per row of a warp's 32 x 32 output patch
constexpr int PF_SMEM = PF_STAGES * (PF_BM * PF_BK + PF_BN * PF_BK) + PF_SRING * PF_SG * 1024 + 1024 /* barriers */ +
                        PF_EPI_WARPS * 32 * PF_PATCH_LD * 4 + 1024 /* alignment slack */;
static_assert(PF_SMEM <= 232448, "shared memory per CTA");

enum { PF_EPI_STORE = 0, PF_EPI_QKV = 1, PF_EPI_RESID = 2, PF_EPI_SWIGLU = 3 };

struct PrefillGemmArgs {
    const float *wsT;  // [K/GS][N]  weight scales, group-major (transposed at load)
    const float *xsT;  // [K/GS][Tpad] activation scales, group-major
    int T, Tpad, N, K;
    float *out;        // STORE: [T][N]; RESID: x[T][N] += ; SWIGLU: hb[T][N/2]
    int ld_out;
    // QKV epilogue
    float *q;          // [T][AH]
    float *kc, *vc;    // layer base of the caches [seq][KV]
    int AH, KV, pos0;
};

__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t saddr) {
    // K-major, SWIZZLE_128B: 8-row atoms of 128 B, atoms 1024 B apart (SBO), LBO unused (=1), version 1
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ULL << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ULL << 46) | (2ULL << 61);
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait_spin(uint64_t *bar, uint32_t parity) {
    long long t0 = clock64();
    unsigned spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 1023u) == 0 && clock64() - t0 > 4000000000LL) __trap(); // never hang the GPU
    }
}
// The epilogue's waits, on 32-bit shared addresses and without a clock read on the fast path (the drain loop is
// instruction-issue bound: the clock-guarded form above costs ~12 instructions per wait even when the barrier is already
// complete).  A failed try_wait suspends the warp in hardware for a while, so the spin bound is seconds, not forever.
__device__ __forceinline__ void pf_wait(uint32_t bar, uint32_t parity) {
    uint32_t n = 0;
    while (true) {
        uint32_t ok;
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok)
                     : "r"(bar), "r"(parity)
                     : "memory");
        if (ok) break;
        if (++n > (1u << 22)) __trap(); // never hang the GPU
    }
}
// One try, result consumed later: the ~100-250 clk a try_wait takes even on a completed barrier then overlap with whatever is
// scheduled between the try and the use of its result.
__device__ __forceinline__ uint32_t pf_try(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    return ok;
}
// one lane of a CONVERGED warp (always the same one): the single-thread tcgen05 / TMA instructions are issued under this predicate
// while the loop around them stays warp-uniform -- inside a divergent `if (lane == 0)` every operand of a uniform-datapath
// instruction (UTCIMMA, UTCBAR, UTMALDG) has to be re-broadcast through an ELECT / R2UR / BRA.U.ANY loop (~8 instructions each)
__device__ __forceinline__ bool pf_elect() {
    uint32_t pred;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void pf_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ float4 lds128f(uint32_t saddr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(saddr));
    return r;
}
#define PF_LD16(d, taddr)                                                                                                            \
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"            \
                 : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(d[4]), "=r"(d[5]), "=r"(d[6]), "=r"(d[7]), "=r"(d[8]),        \
                   "=r"(d[9]), "=r"(d[10]), "=r"(d[11]), "=r"(d[12]), "=r"(d[13]), "=r"(d[14]), "=r"(d[15])                           \
                 : "r"(taddr)                                                                                                        \
                 : "memory")
__device__ __forceinline__ void pf_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 16 accumulator columns of one group: acc[j] += (f32(dot_j) * ws_j) * xs.
// EXACT: unfused multiplies and add, i.e. the reference's left fold term by term (tensor.rs:59-61) -- bit-identical.
// fast: the same exact int32 dots; p = ws * xs is formed first (it does not depend on the TMEM read), then one packed FMA.
template <bool EXACT>
__device__ __forceinline__ void pf_scale16(float *acc, const uint32_t (&d)[16], uint32_t ws_saddr, float xs) {
    const float2 xs2 = make_float2(xs, xs);
#pragma unroll
    for (int j4 = 0; j4 < 4; j4++) {
        const float4 w = lds128f(ws_saddr + 16 * j4);
        if (EXACT) {
            acc[4 * j4 + 0] = __fadd_rn(acc[4 * j4 + 0], __fmul_rn(__fmul_rn((float)(int)d[4 * j4 + 0], w.x), xs));
            acc[4 * j4 + 1] = __fadd_rn(acc[4 * j4 + 1], __fmul_rn(__fmul_rn((float)(int)d[4 * j4 + 1], w.y), xs));
            acc[4 * j4 + 2] = __fadd_rn(acc[4 * j4 + 2], __fmul_rn(__fmul_rn((float)(int)d[4 * j4 + 2], w.z), xs));
            acc[4 * j4 + 3] = __fadd_rn(acc[4 * j4 + 3], __fmul_rn(__fmul_rn((float)(int)d[4 * j4 + 3], w.w), xs));
        } else {
            float2 *ac = reinterpret_cast<float2 *>(acc + 4 * j4);
            const float2 p01 = __fmul2_rn(make_float2(w.x, w.y), xs2), p23 = __fmul2_rn(make_float2(w.z, w.w), xs2);
            ac[0] = __ffma2_rn(make_float2((float)(int)d[4 * j4 + 0], (float)(int)d[4 * j4 + 1]), p01, ac[0]);
            ac[1] = __ffma2_rn(make_float2((float)(int)d[4 * j4 + 2], (float)(int)d[4 * j4 + 3]), p23, ac[1]);
        }
    }
}

// Shared-memory layout of k_gemm_q8 as byte offsets from the 1 KB-aligned base: every address the hot loops use is base + constant
constexpr uint32_t PF_OFF_A = 0;                                                 // [STAGES][128 rows][128 B] activation tiles
constexpr uint32_t PF_OFF_B = PF_STAGES * PF_BM * PF_BK;                         // [STAGES][128 rows][128 B] weight tiles
constexpr uint32_t PF_OFF_SCALE = PF_STAGES * (PF_BM + PF_BN) * PF_BK;           // [PF_SRING][ws g0 | ws g1 | xs g0 | xs g1] x 128 f32
constexpr uint32_t PF_OFF_BAR = PF_OFF_SCALE + PF_SRING * PF_SG * 1024;          // mbarriers (8 B each), then the TMEM base slot
constexpr uint32_t PF_BAR_FULL = PF_OFF_BAR, PF_BAR_EMPTY = PF_BAR_FULL + 8 * PF_STAGES, PF_BAR_TFULL = PF_BAR_EMPTY + 8 * PF_STAGES,
                   PF_BAR_TEMPTY = PF_BAR_TFULL + 16 /* [2 pair slots][2 groups] */, PF_BAR_SFULL = PF_BAR_TEMPTY + 32,
                   PF_BAR_SEMPTY = PF_BAR_SFULL + 8 * PF_SRING, PF_OFF_TMEM = PF_BAR_SEMPTY + 8 * PF_SRING;
constexpr uint32_t PF_OFF_PATCH = PF_OFF_BAR + 1024;                             // [16 warps][32 rows][PF_PATCH_LD] f32 output patches
static_assert(PF_OFF_TMEM + 4 <= PF_OFF_PATCH, "barrier block");
static_assert(PF_OFF_PATCH + PF_EPI_WARPS * 32 * PF_PATCH_LD * 4 + 1024 <= PF_SMEM, "shared memory budget");

__device__ __forceinline__ void sts128f(uint32_t saddr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Drain one accumulator PAIR (two quantisation groups) of this thread's 32 columns, as a stream of 16-column chunks through
// two register buffers: the TMEM read of the next chunk is always in flight while the current one is being scaled.  The
// stream does not stop at the pair boundary -- the first chunk of this pair (d0) was requested while the previous pair was
// being finished, and before the last chunk is scaled the first chunk of the NEXT pair (nxt_taddr, possibly of the next tile)
// is requested; whether that pair is complete is asked (try_wait) one scaling block earlier and looked at only then, so
// neither the barrier latency nor a TMEM read latency sits exposed between two pairs.  Each group accumulator goes back to the
// MMA warp as soon as its second chunk has landed in registers (group 0 two scaling blocks before group 1).
// ws0 / xsa: shared addresses of this thread's 32 weight scales / its token scale for the pair's first group (the second group's
// follow 512 B later).  tempty_bar: the slot's two "drained" barriers (group 0, group 1).
template <bool EXACT>
__device__ __forceinline__ void pf_drain_pair(float (&acc)[PF_COLS], uint32_t (&d0)[16], uint32_t (&d1)[16], uint32_t taddr, uint32_t ws0, uint32_t xsa,
                                              uint32_t tempty_bar, int lane, uint32_t nxt_taddr, uint32_t nxt_bar, uint32_t nxt_parity) {
    const float xs = lds_f32(xsa);
    pf_wait_ld(); // d0 = group 0, columns 0..15
    PF_LD16(d1, taddr + 16);
    pf_scale16<EXACT>(acc, d0, ws0, xs);
    pf_wait_ld();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) pf_arrive(tempty_bar); // group 0 of the pair is in registers: its accumulator may be refilled already
    PF_LD16(d0, taddr + PF_BN);
    const float xsb = lds_f32(xsa + 512);
    pf_scale16<EXACT>(acc + 16, d1, ws0 + 64, xs);
    pf_wait_ld();
    PF_LD16(d1, taddr + PF_BN + 16);
    const uint32_t nxt_ok = pf_try(nxt_bar, nxt_parity); // asked now, looked at after the scaling block below
    pf_scale16<EXACT>(acc, d0, ws0 + 512, xsb);
    pf_wait_ld();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) pf_arrive(tempty_bar + 8); // group 1 drained into registers
    if (!nxt_ok) pf_wait(nxt_bar, nxt_parity);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    PF_LD16(d0, nxt_taddr); // first chunk of the next pair: in flight while the last chunk of this one is scaled
    pf_scale16<EXACT>(acc + 16, d1, ws0 + 512 + 64, xsb);
}

// EXACT = false: the fast drain (what q3_prefill runs): the exact int32 group dots, folded with packed f32x2 FMAs.
// EXACT = true: every output is the reference's left fold of unfused (dot * ws) * xs terms -- bit-identical to `matmul`
//               (the operator-level proof).
// K / GS must be even (checked by the host): the unit of hand-over between the MMA warp and the epilogue is a PAIR of group
// accumulators (2 x 128 TMEM columns; two pair slots fill the 512 columns), and a scale-ring slot holds the rows of one pair.
// PERSISTENT: grid = min(tiles, SMs); a CTA walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... (token tile fastest, so the
// CTAs running together share weight tiles in L2).  The TMA and MMA warps run straight on into the next tile (stage ring,
// accumulator pairs and scale ring keep their running indices), so a tile's output store and the pipeline refill overlap
// and TMEM is allocated once per SM instead of once per tile.
template <int GS, int EPI, bool EXACT>
__global__ void __launch_bounds__(PF_THREADS, 1) // 96 registers: three schedulers host 5 warps (16384 / (5 x 32) = 102; 112 does not launch)
    k_gemm_q8(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_xs,
              const __grid_constant__ CUtensorMap map_ws, const PrefillGemmArgs a) {
    extern __shared__ __align__(1024) uint8_t pf_smem_raw[];
    uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(pf_smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t sb = smem_u32(smem); // every shared address below is sb + a constant
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mt = a.Tpad / PF_BM, ntile = mt * (a.N / PF_BN);
    const int nkb = a.K / PF_BK;
    constexpr int GPS = PF_BK / GS; // groups per stage
    constexpr int KPG = GS / 32;    // MMA K-steps per group
    const int npair = (a.K / GS) >> 1; // accumulator pairs per tile
    static_assert(PF_NACC == 4 && PF_SG == 2 && (PF_SRING & (PF_SRING - 1)) == 0, "pairs");

    if (threadIdx.x == 0) {
        for (int s = 0; s < PF_STAGES; s++) {
            mbar_init(reinterpret_cast<uint64_t *>(smem + PF_BAR_FULL) + s, 1);
            mbar_init(reinterpret_cast<uint64_t *>(smem + PF_BAR_EMPTY) + s, 1);
        }
        for (int b = 0; b < 2; b++) mbar_init(reinterpret_cast<uint64_t *>(smem + PF_BAR_TFULL) + b, 1);
        for (int b = 0; b < 4; b++) mbar_init(reinterpret_cast<uint64_t *>(smem + PF_BAR_TEMPTY) + b, PF_EPI_WARPS); // one arrive per epilogue warp
        for (int b = 0; b < PF_SRING; b++) {
            mbar_init(reinterpret_cast<uint64_t *>(smem + PF_BAR_SFULL) + b, 1);
            mbar_init(reinterpret_cast<uint64_t *>(smem + PF_BAR_SEMPTY) + b, PF_EPI_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_xs) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ws) : "memory");
    }
    if (warp == PF_MMA_WARP) { // TMEM: all 512 columns = 2 pairs of 128 x 128 int32 accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sb + PF_OFF_TMEM), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *reinterpret_cast<uint32_t *>(smem + PF_OFF_TMEM);

    if (warp == PF_TMA_WARP) {
        // ------------------------------- tile producer (whole warp runs the loop, one elected lane issues) -------------------------------
        int kbt = 0; // running stage uses across tiles
        for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
            const int m0 = (tile % mt) * PF_BM, n0 = (tile / mt) * PF_BN;
            for (int kb = 0; kb < nkb; kb++, kbt++) {
                const int s = kbt % PF_STAGES;
                pf_wait(sb + PF_BAR_EMPTY + 8 * s, ((kbt / PF_STAGES) & 1) ^ 1);
                if (pf_elect()) {
                    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + PF_BAR_FULL) + s;
                    mbar_expect_tx(bar, (PF_BM + PF_BN) * PF_BK);
                    tma_load_2d(smem + PF_OFF_A + (size_t)s * PF_BM * PF_BK, &map_x, kb * PF_BK, m0, bar);
                    tma_load_2d(smem + PF_OFF_B + (size_t)s * PF_BN * PF_BK, &map_w, kb * PF_BK, n0, bar);
                }
                __syncwarp();
            }
        }
    } else if (warp == PF_SCALE_WARP) {
        // ------------------------------- scale-row producer -------------------------------
        // The scale rows of an accumulator pair (2 groups x 128 weight scales, 2 groups x 128 token scales: two tensor copies) go
        // through their own ring, fed by their own warp: it runs as far ahead of the epilogue as the ring is deep (PF_SRING pairs,
        // across tile boundaries), independent of the tile producer.  History: as eight 512-byte bulk copies per stage issued by the
        // tile producer from a divergent single-lane branch, the scale traffic -- not the tensor pipe, not the epilogue -- set the
        // pace of the whole kernel (8B gate/up: 650 us; the same kernel with the scale traffic switched off: 457 us).
        int sc = 0; // running pair count
        for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
            const int m0 = (tile % mt) * PF_BM, n0 = (tile / mt) * PF_BN;
            for (int c = 0; c < npair; c++, sc++) {
                const int sl = sc & (PF_SRING - 1);
                pf_wait(sb + PF_BAR_SEMPTY + 8 * sl, ((sc / PF_SRING) & 1) ^ 1);
                if (pf_elect()) {
                    uint64_t *bar = reinterpret_cast<uint64_t *>(smem + PF_BAR_SFULL) + sl;
                    mbar_expect_tx(bar, 2048);
                    tma_load_2d(smem + PF_OFF_SCALE + sl * 2048, &map_ws, n0, 2 * c, bar);
                    tma_load_2d(smem + PF_OFF_SCALE + sl * 2048 + 1024, &map_xs, m0, 2 * c, bar);
                }
                __syncwarp();
            }
        }
    } else if (warp == PF_MMA_WARP) {
        // ------------------------------- MMA issuer (whole warp runs the loop, one elected lane issues) -------------------------------
        // instruction descriptor: D = S32, A = B = signed int8, both K-major, N = 128, M = 128
        constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((PF_BN >> 3) << 17) | ((PF_BM >> 4) << 24);
        uint64_t *tfull = reinterpret_cast<uint64_t *>(smem + PF_BAR_TFULL), *empty = reinterpret_cast<uint64_t *>(smem + PF_BAR_EMPTY);
        int kbt = 0, pt = 0; // running stage uses, accumulator-pair uses
        const uint64_t desc_a0 = umma_desc_k_sw128(sb + PF_OFF_A), desc_b0 = umma_desc_k_sw128(sb + PF_OFF_B);
        for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
            int gi = 0;
            for (int kb = 0; kb < nkb; kb++, kbt++) {
                const int s = kbt % PF_STAGES;
                pf_wait(sb + PF_BAR_FULL + 8 * s, (kbt / PF_STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                // descriptors of this stage: the start-address field counts 16-byte units (stages are 16 KB apart, K-steps 32 B)
                const uint64_t da = desc_a0 + (uint64_t)(s * (PF_BM * PF_BK / 16)), db = desc_b0 + (uint64_t)(s * (PF_BN * PF_BK / 16));
#pragma unroll
                for (int gg = 0; gg < GPS; gg++, gi++) {
                    const int ps = pt & 1;
                    // each group accumulator of a pair is handed back on its own: the first one two scaling blocks earlier
                    const uint32_t col = ps * 2 * PF_BN + (gi & 1) * PF_BN;
                    pf_wait(sb + PF_BAR_TEMPTY + 8 * (2 * ps + (gi & 1)), ((pt >> 1) & 1) ^ 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (pf_elect()) {
#pragma unroll
                        for (int kk = 0; kk < KPG; kk++) {
                            const uint32_t koff = (gg * GS + kk * 32) >> 4; // along K inside the 128 B swizzle span, in 16-byte units
                            umma_i8(tmem_base + col, da + koff, db + koff, IDESC, kk > 0);
                        }
                        if (gi & 1) umma_commit(&tfull[ps]); // pair complete -> epilogue
                    }
                    __syncwarp();
                    if (gi & 1) pt++;
                }
                if (pf_elect()) umma_commit(&empty[s]); // all MMAs reading this stage retired -> TMA may refill it
                __syncwarp();
            }
        }
        // one empty pair: the epilogue's last look-ahead waits for it (and reads an accumulator nobody uses)
        if (pf_elect()) umma_commit(&tfull[pt & 1]);
        __syncwarp();
    } else if (warp < PF_EPI_WARPS) {
        // ------------------------------- epilogue -------------------------------
        const int quad = warp & 3;  // TMEM lanes [32*quad, 32*quad+32) are the only ones this warp may read
        const int part = warp >> 2; // which PF_COLS accumulator columns
        const uint32_t tq = tmem_base + ((uint32_t)(quad * 32) << 16) + part * PF_COLS;
        const uint32_t wsx = sb + PF_OFF_SCALE + part * (PF_COLS * 4);                 // this thread's weight scales in scale slot 0, row 0
        const uint32_t xsx = sb + PF_OFF_SCALE + 1024 + (quad * 32 + lane) * 4;        // its token scale (slot: ws g0 | ws g1 | xs g0 | xs g1)
        int pt = 0;                 // running pair count (pair slot = pt & 1, scale slot = pt & (PF_SRING - 1))
        uint32_t d0[16], d1[16];    // the two chunk buffers of the TMEM read stream (live across pairs and tiles)
        uint32_t s_ok = 0;          // the scale rows of the pair about to start are known to have landed (asked ahead of time)
        // the very first pair of this CTA: nobody has requested its first chunk yet
        pf_wait(sb + PF_BAR_TFULL, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        PF_LD16(d0, tq);
        for (int tile = blockIdx.x; tile < ntile; tile += gridDim.x) {
            float acc[PF_COLS];
#pragma unroll
            for (int j = 0; j < PF_COLS; j++) acc[j] = 0.0f;
#pragma unroll 1
            for (int c = 0; c < npair; c++, pt++) {
                const uint32_t ps = pt & 1, sl = pt & (PF_SRING - 1);
                if (!s_ok) pf_wait(sb + PF_BAR_SFULL + 8 * sl, (pt / PF_SRING) & 1); // the pair's scale rows landed
                // the next pair's scale rows: asked for here, looked at when they are needed (never, after the very last pair)
                s_ok = pf_try(sb + PF_BAR_SFULL + 8 * ((pt + 1) & (PF_SRING - 1)), ((pt + 1) / PF_SRING) & 1);
                pf_drain_pair<EXACT>(acc, d0, d1, tq + ps * (2 * PF_BN), wsx + sl * 2048, xsx + sl * 2048, sb + PF_BAR_TEMPTY + 16 * ps, lane,
                                     tq + (ps ^ 1) * (2 * PF_BN), sb + PF_BAR_TFULL + 8 * (ps ^ 1), ((pt + 1) >> 1) & 1);
                __syncwarp();
                if (lane == 0) pf_arrive(sb + PF_BAR_SEMPTY + 8 * sl); // scale rows consumed
            }
            // ---- write the tile out ----
            // A thread owns a token ROW (TMEM lane) and 32 consecutive columns, so direct stores would touch 32 different cache
            // lines per warp instruction (measured: ~8 700 clk per tile, 15 % of the tile, in the in-kernel trace).  Each warp
            // therefore turns its 32 x 32 block through a private shared-memory patch (pitch 36 floats: conflict-free for the
            // 128-bit stores and loads) and writes 4 full 128-byte row segments per instruction.
            {
                const int m0 = (tile % mt) * PF_BM, n0 = (tile / mt) * PF_BN;
                const uint32_t patch = sb + PF_OFF_PATCH + warp * (32 * PF_PATCH_LD * 4);
#pragma unroll
                for (int j4 = 0; j4 < PF_COLS / 4; j4++)
                    sts128f(patch + (lane * PF_PATCH_LD + 4 * j4) * 4, make_float4(acc[4 * j4], acc[4 * j4 + 1], acc[4 * j4 + 2], acc[4 * j4 + 3]));
                __syncwarp();
                const int r4 = lane >> 3, c4 = lane & 7;
                const int c0 = n0 + part * PF_COLS; // first column of the warp's block
                float *base; // row pointer of token 0 for this block, and the row pitch
                int ld;
                if (EPI == PF_EPI_STORE || EPI == PF_EPI_RESID) { base = a.out + c0; ld = a.ld_out; }
                else if (EPI == PF_EPI_SWIGLU) { base = a.out + c0 / 2; ld = a.ld_out; }
                else if (c0 < a.AH) { base = a.q + c0; ld = a.AH; } // PF_EPI_QKV: rows [0,AH) -> q[t], [AH,AH+KV) -> K cache row pos0+t, then V (layers.rs:334-336)
                else if (c0 < a.AH + a.KV) { base = a.kc + (size_t)a.pos0 * a.KV + (c0 - a.AH); ld = a.KV; }
                else { base = a.vc + (size_t)a.pos0 * a.KV + (c0 - a.AH - a.KV); ld = a.KV; }
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int row = 4 * k + r4, tr = m0 + quad * 32 + row;
                    const float4 v = lds128f(patch + (row * PF_PATCH_LD + 4 * c4) * 4);
                    if (tr < a.T) {
                        if (EPI == PF_EPI_SWIGLU) { // rows interleaved (gate_j, up_j): layers.rs:472-475
                            const float s0 = __fmul_rn(v.x, __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-v.x))));
                            const float s1 = __fmul_rn(v.z, __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-v.z))));
                            *reinterpret_cast<float2 *>(base + (size_t)tr * ld + 2 * c4) = make_float2(__fmul_rn(s0, v.y), __fmul_rn(s1, v.w));
                        } else {
                            float4 *dst = reinterpret_cast<float4 *>(base + (size_t)tr * ld + 4 * c4);
                            if (EPI == PF_EPI_RESID) { // x += (layers.rs:249-259)
                                const float4 o = *dst;
                                *dst = make_float4(__fadd_rn(o.x, v.x), __fadd_rn(o.y, v.y), __fadd_rn(o.z, v.z), __fadd_rn(o.w, v.w));
                            } else {
                                *dst = v;
                            }
                        }
                    }
                }
                __syncwarp(); // the patch is rewritten at the end of the next tile
            }
        }
        pf_wait_ld(); // the stream's last look-ahead read
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == PF_MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}
#undef PF_LD16

// ------------------------------------------------------------------------------------------
// batched helpers around the GEMM
// ------------------------------------------------------------------------------------------
// per-token RMSNorm (+ embedding gather) + group quantise; scales written group-major [ng][Tpad].
// grid = T, block = 256.  (layers.rs:72-76, 109-130; tensor.rs:91-119)
// MAXV: float4 per thread held in registers (n <= 1024 * MAXV): 4 covers every dim <= 4096 at 16 registers instead of 64 --
// 8 resident blocks per SM instead of 3 (the kernel is latency-bound: load -> reduce -> quantise per token).
template <int GS, int MAXV = 16>
__global__ void __launch_bounds__(256) k_pf_norm_quant(float *x, const float *w, int8_t *q, float *sT, int n, int Tpad,
                                                       const int8_t *embed_q, const float *embed_s, const int *tokens, int write_normed) {
    __shared__ float red[8];
    __shared__ float s_f;
    const int t = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float *xr = x + (size_t)t * n;
    const int n4 = n >> 2;
    float4 v[MAXV];
    float ss = 0.0f;
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        int i4 = tid + k * 256;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i4 < n4) {
            if (embed_q) {
                size_t base = (size_t)tokens[t] * n + (size_t)i4 * 4;
                char4 e = *reinterpret_cast<const char4 *>(embed_q + base);
                float sc = embed_s[base / GS];
                v[k] = make_float4((float)e.x * sc, (float)e.y * sc, (float)e.z * sc, (float)e.w * sc);
                reinterpret_cast<float4 *>(xr)[i4] = v[k];
            } else {
                v[k] = reinterpret_cast<const float4 *>(xr)[i4];
            }
            ss += __fmul_rn(v[k].x, v[k].x);
            ss += __fmul_rn(v[k].y, v[k].y);
            ss += __fmul_rn(v[k].z, v[k].z);
            ss += __fmul_rn(v[k].w, v[k].w);
        }
    }
    ss = warp_sum(ss);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    if (tid == 0) {
        float tsum = 0.0f;
        for (int i = 0; i < 8; i++) tsum += red[i];
        s_f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(tsum, (float)n), NORM_EPS)));
    }
    __syncthreads();
    const float f = s_f;
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        int i4 = tid + k * 256;
        if (i4 - lane < n4) {
            float4 y = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i4 < n4) {
                float4 wv = __ldg(reinterpret_cast<const float4 *>(w) + i4);
                y.x = __fmul_rn(wv.x, __fmul_rn(f, v[k].x));
                y.y = __fmul_rn(wv.y, __fmul_rn(f, v[k].y));
                y.z = __fmul_rn(wv.z, __fmul_rn(f, v[k].z));
                y.w = __fmul_rn(wv.w, __fmul_rn(f, v[k].w));
            }
            uint32_t packed;
            float scale;
            quantize_group4<GS>(y, packed, scale);
            if (i4 < n4) {
                reinterpret_cast<uint32_t *>(q + (size_t)t * n)[i4] = packed;
                if ((i4 % (GS / 4)) == 0) sT[(size_t)(i4 / (GS / 4)) * Tpad + t] = scale;
                if (write_normed) reinterpret_cast<float4 *>(xr)[i4] = y;
            }
        }
    }
}

// per-token group quantise of [T][n] f32; scales group-major.  grid = T.
template <int GS>
__global__ void __launch_bounds__(256) k_pf_quantize(const float *__restrict__ x, int8_t *q, float *sT, int n, int Tpad) {
    const int t = blockIdx.x, lane = threadIdx.x & 31;
    const int n4 = n >> 2;
    const float *xr = x + (size_t)t * n;
    for (int base = threadIdx.x - lane; base < n4; base += 256) {
        int i4 = base + lane;
        float4 y = (i4 < n4) ? reinterpret_cast<const float4 *>(xr)[i4] : make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t packed;
        float scale;
        quantize_group4<GS>(y, packed, scale);
        if (i4 < n4) {
            reinterpret_cast<uint32_t *>(q + (size_t)t * n)[i4] = packed;
            if ((i4 % (GS / 4)) == 0) sT[(size_t)(i4 / (GS / 4)) * Tpad + t] = scale;
        }
    }
}

// QK-norm + RoPE for T tokens: grid = (ceil((n_heads + n_kv)/4), T), block 128 (one warp per head).
__global__ void __launch_bounds__(128) k_pf_qknorm_rope(float *q, float *kc_layer, const float *q_ln, const float *k_ln,
                                                        const float *rope, int pos0, int n_heads, int n_kv, int AH, int KV) {
    const int lane = threadIdx.x & 31;
    const int head = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int t = blockIdx.y;
    if (head >= n_heads + n_kv) return;
    const int pos = pos0 + t;
    float *p = head < n_heads ? q + (size_t)t * AH + (size_t)head * HEAD_DIM
                              : kc_layer + (size_t)pos * KV + (size_t)(head - n_heads) * HEAD_DIM;
    float4 v = reinterpret_cast<float4 *>(p)[lane];
    float4 r = qk_norm_rope(v, head < n_heads ? q_ln : k_ln, rope + (size_t)pos * HEAD_DIM, lane);
    reinterpret_cast<float4 *>(p)[lane] = r;
}

// ------------------------------------------------------------------------------------------
// Causal attention for T query tokens over the cache (key positions 0..pos0+t for query t; layers.rs:374-419 with an online
// softmax) on the tensor cores: mma.sync m16n8k16 on an FP16 hi / lo split with f32 accumulation.
//   x = hi + lo, hi = fp16(x), lo = fp16(x - hi);  a*b ~ hi*hi + hi*lo + lo*hi   (relative error ~2^-21 instead of 2^-11 for a
//   single FP16 or TF32 product: the attention output is re-quantised to int8 right after, and a coarser score would flip far
//   more int8 values than f32 arithmetic does).
// FP16 rather than TF32 operands: a k16 MMA covers twice the depth of a TF32 k8 one (half the MMA count), the operands are half
// as wide in shared memory, and fragments come in with ldmatrix (4 8x8 tiles per instruction instead of 32-bit loads).  K / V
// are split ONCE per layer by k_pf_split_kv rather than by every CTA that streams them -- the tiles then arrive with cp.async,
// double-buffered, no ALU work on the way.
//   FP16 range: hi overflows beyond 65504 (K is QK-normalised, P <= 1; V / Q of that size do not occur), and a lo part below
//   6.1e-5 is subnormal -- an absolute error of <= 3e-8 per element, far below the f32 round-off of the sums it enters.
// One CTA = one kv head x 64 query rows (64 / KVMUL tokens x the KVMUL heads that share the K / V stream), 4 warps x 16 rows,
// key tiles of 32 positions.  Shared memory rows are 128 halfs = 256 B = 16 chunks of 16 B; chunk c of row r sits at chunk
// c ^ (r & 7), which makes every ldmatrix phase (8 rows, same logical chunk) conflict-free.
//   S = Q K^T : A = Q (ldmatrix), B = K rows as stored (ldmatrix, non-transposed: a K row IS a column of K^T)
//   O += P V  : A = P straight from the S accumulators (two adjacent 8-key tiles form one k16 fragment), B = V (ldmatrix.trans)
// ------------------------------------------------------------------------------------------
constexpr int PFH_R = 64, PFH_BK = 32;
constexpr int PFH_SMEM = 2 * PFH_R * HEAD_DIM * 2 + 2 * 4 * PFH_BK * HEAD_DIM * 2; // Q hi/lo + 2 stages x (K hi, K lo, V hi, V lo) = 96 KB

// rows [0, rows) of one layer's K and V cache (f32 [rows][KV]) -> hi / lo halves, four arrays [rows][KV]: Kh | Kl | Vh | Vl
__global__ void __launch_bounds__(256) k_pf_split_kv(const float *__restrict__ kc, const float *__restrict__ vc, __half *out, size_t n4, size_t plane) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < 2 * n4; i += (size_t)gridDim.x * blockDim.x) {
        const bool isv = i >= n4;
        const size_t j = isv ? i - n4 : i;
        const float4 x = reinterpret_cast<const float4 *>(isv ? vc : kc)[j];
        const __half2 h0 = __floats2half2_rn(x.x, x.y), h1 = __floats2half2_rn(x.z, x.w);
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        const __half2 l0 = __floats2half2_rn(__fsub_rn(x.x, f0.x), __fsub_rn(x.y, f0.y)), l1 = __floats2half2_rn(__fsub_rn(x.z, f1.x), __fsub_rn(x.w, f1.y));
        __half *dst = out + (isv ? 2 * plane : 0) + 4 * j;
        *reinterpret_cast<uint2 *>(dst) = make_uint2(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1));
        *reinterpret_cast<uint2 *>(dst + plane) = make_uint2(*reinterpret_cast<const uint32_t *>(&l0), *reinterpret_cast<const uint32_t *>(&l1));
    }
}

__device__ __forceinline__ void mma_f16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm4(uint32_t (&r)[4], uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void ldsm4t(uint32_t (&r)[4], uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void pfh_split2(float x, float y, uint32_t &hi, uint32_t &lo) {
    const __half2 h = __floats2half2_rn(x, y);
    const float2 f = __half22float2(h);
    const __half2 l = __floats2half2_rn(__fsub_rn(x, f.x), __fsub_rn(y, f.y));
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}

// kvh: [4][rows_alloc][KV] halves from k_pf_split_kv (plane = rows_alloc * KV)
template <int KVMUL>
__global__ void __launch_bounds__(128, 2) k_pf_attention_h(const float *__restrict__ q, const __half *__restrict__ kvh, size_t plane, float *out, int T,
                                                           int pos0, int AH, int KV) {
    extern __shared__ __align__(1024) uint8_t pfh_smem[];
    const uint32_t sQ = smem_u32(pfh_smem);                      // Qh [64][128] | Ql [64][128]
    const uint32_t sKV = sQ + 2 * PFH_R * HEAD_DIM * 2;          // [2 stages][Kh | Kl | Vh | Vl][32][128]
    constexpr uint32_t QL = PFH_R * HEAD_DIM * 2, ARR = PFH_BK * HEAD_DIM * 2, STAGE = 4 * ARR;
    constexpr int BQ = PFH_R / KVMUL;
    // the query tiles with the longest causal horizon are launched first (a late tile does up to T / 64 times the work of the first)
    const int kvhd = blockIdx.x, q0 = ((int)gridDim.y - 1 - (int)blockIdx.y) * BQ;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
    const float scale = __fdiv_rn(1.0f, sqrtf((float)HEAD_DIM));
    int last_q = q0 + BQ - 1;
    if (last_q > T - 1) last_q = T - 1;
    const int nkeys = pos0 + last_q + 1; // causal horizon of the last query in the tile
    const int ntiles = (nkeys + PFH_BK - 1) / PFH_BK;

    // stage loader: 4 arrays x 32 rows x 16 chunks = 2048 16-byte copies, 16 per thread; rows past the horizon are zero-filled
    auto load_stage = [&](int tile, int st) {
        const int k0 = tile * PFH_BK;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const int idx = tid + i * 128, arr = idx >> 9, p = (idx >> 4) & 31, c = idx & 15;
            const int key = k0 + p;
            const bool ok = key < nkeys;
            const __half *src = kvh + (size_t)arr * plane + (size_t)(ok ? key : 0) * KV + (size_t)kvhd * HEAD_DIM + c * 8;
            const uint32_t dst = sKV + st * STAGE + arr * ARR + p * 256 + ((c ^ (p & 7)) << 4);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(ok ? 16 : 0) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    load_stage(0, 0);
    // Q tile: row r <-> (token q0 + r / KVMUL, head kvhd*KVMUL + r % KVMUL), split once
    for (int i = tid; i < PFH_R * 16; i += 128) {
        const int r = i >> 4, c = i & 15;
        const int tq = q0 + r / KVMUL;
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
        if (tq < T) {
            const float4 *src = reinterpret_cast<const float4 *>(q + (size_t)tq * AH + (size_t)(kvhd * KVMUL + r % KVMUL) * HEAD_DIM + c * 8);
            v0 = src[0];
            v1 = src[1];
        }
        uint32_t h[4], l[4];
        pfh_split2(v0.x, v0.y, h[0], l[0]);
        pfh_split2(v0.z, v0.w, h[1], l[1]);
        pfh_split2(v1.x, v1.y, h[2], l[2]);
        pfh_split2(v1.z, v1.w, h[3], l[3]);
        const uint32_t off = r * 256 + ((c ^ (r & 7)) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(sQ + off), "r"(h[0]), "r"(h[1]), "r"(h[2]), "r"(h[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(sQ + QL + off), "r"(l[0]), "r"(l[1]), "r"(l[2]), "r"(l[3]) : "memory");
    }
    const int r0 = warp * 16 + g, r1 = r0 + 8;                                   // this thread's two rows of the tile
    const int qp0 = pos0 + q0 + r0 / KVMUL, qp1 = pos0 + q0 + r1 / KVMUL;          // their absolute positions
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.0f, l1 = 0.0f;
    float o[16][4];
#pragma unroll
    for (int j = 0; j < 16; j++) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.0f;
    // ldmatrix lane roles
    const int a_row = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, a_cg = (lane >> 4) & 1;      // A (Q): row, which 8-column half of the k16 step
    const int b_key = (lane & 7) + ((lane >> 4) & 1) * 8, b_cg = (lane >> 3) & 1;                  // B (K): key within a 16-key group, 8-dim half
    const int v_key = (lane & 7) + ((lane >> 3) & 1) * 8, v_cg = (lane >> 4) & 1;                  // B (V, transposed): key within the k16 step, 8-dim half

    for (int tile = 0; tile < ntiles; tile++) {
        const int st = tile & 1, k0 = tile * PFH_BK;
        if (tile + 1 < ntiles) {
            load_stage(tile + 1, st ^ 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads(); // tile `tile` (and, first time round, the Q tile) visible to every warp
        const uint32_t sKh = sKV + st * STAGE, sKl = sKh + ARR, sVh = sKh + 2 * ARR, sVl = sKh + 3 * ARR;
        // ---- S = Q K^T (16 rows x 32 keys per warp) ----
        float s[4][4];
#pragma unroll
        for (int j = 0; j < 4; j++) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.0f;
#pragma unroll
        for (int ks = 0; ks < 8; ks++) {
            uint32_t ah[4], al[4];
            const uint32_t aoff = a_row * 256 + (((2 * ks + a_cg) ^ (a_row & 7)) << 4);
            ldsm4(ah, sQ + aoff);
            ldsm4(al, sQ + QL + aoff);
            // the three product terms go round the four key tiles: consecutive MMAs never touch the same accumulator
            uint32_t bh[2][4], bl[2][4];
#pragma unroll
            for (int jj = 0; jj < 2; jj++) { // 16 keys per ldmatrix.x4: n-tiles 2jj, 2jj+1
                const int key = 16 * jj + b_key;
                const uint32_t boff = key * 256 + (((2 * ks + b_cg) ^ (key & 7)) << 4);
                ldsm4(bh[jj], sKh + boff);
                ldsm4(bl[jj], sKl + boff);
            }
#pragma unroll
            for (int j = 0; j < 4; j++) mma_f16(s[j], al[0], al[1], al[2], al[3], bh[j >> 1][2 * (j & 1)], bh[j >> 1][2 * (j & 1) + 1]);
#pragma unroll
            for (int j = 0; j < 4; j++) mma_f16(s[j], ah[0], ah[1], ah[2], ah[3], bl[j >> 1][2 * (j & 1)], bl[j >> 1][2 * (j & 1) + 1]);
#pragma unroll
            for (int j = 0; j < 4; j++) mma_f16(s[j], ah[0], ah[1], ah[2], ah[3], bh[j >> 1][2 * (j & 1)], bh[j >> 1][2 * (j & 1) + 1]);
        }
        // ---- online softmax: thread holds keys k0 + 8j + {2t, 2t+1} of rows r0 (s[j][0..1]) and r1 (s[j][2..3]) ----
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int key = k0 + 8 * j + 2 * t;
            s[j][0] = (key <= qp0) ? __fmul_rn(s[j][0], scale) : -INFINITY;
            s[j][1] = (key + 1 <= qp0) ? __fmul_rn(s[j][1], scale) : -INFINITY;
            s[j][2] = (key <= qp1) ? __fmul_rn(s[j][2], scale) : -INFINITY;
            s[j][3] = (key + 1 <= qp1) ? __fmul_rn(s[j][3], scale) : -INFINITY;
            mx0 = fmaxf(mx0, fmaxf(s[j][0], s[j][1]));
            mx1 = fmaxf(mx1, fmaxf(s[j][2], s[j][3]));
        }
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
        mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
        mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
        const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
        const float c0 = (mn0 == -INFINITY) ? 1.0f : expf(m0 - mn0), c1 = (mn1 == -INFINITY) ? 1.0f : expf(m1 - mn1);
        m0 = mn0;
        m1 = mn1;
        l0 *= c0;
        l1 *= c1;
#pragma unroll
        for (int j = 0; j < 16; j++) {
            o[j][0] *= c0;
            o[j][1] *= c0;
            o[j][2] *= c1;
            o[j][3] *= c1;
        }
        // ---- O += P V: k16 step kk = keys 16kk .. 16kk+15 = S tiles 2kk, 2kk+1 ----
#pragma unroll
        for (int kk = 0; kk < 2; kk++) {
            uint32_t ph[4], pl[4];
#pragma unroll
            for (int h2 = 0; h2 < 2; h2++) {
                const float *sj = s[2 * kk + h2];
                const float p00 = (sj[0] == -INFINITY) ? 0.0f : expf(sj[0] - mn0), p01 = (sj[1] == -INFINITY) ? 0.0f : expf(sj[1] - mn0);
                const float p10 = (sj[2] == -INFINITY) ? 0.0f : expf(sj[2] - mn1), p11 = (sj[3] == -INFINITY) ? 0.0f : expf(sj[3] - mn1);
                l0 += p00 + p01;
                l1 += p10 + p11;
                pfh_split2(p00, p01, ph[2 * h2], pl[2 * h2]);         // a0a1 / a4a5: row g
                pfh_split2(p10, p11, ph[2 * h2 + 1], pl[2 * h2 + 1]); // a2a3 / a6a7: row g+8
            }
            const int key = 16 * kk + v_key;
#pragma unroll
            for (int n4 = 0; n4 < 4; n4++) { // 32 dims = four output tiles per round, the three product terms go round them
                uint32_t vh[2][4], vl[2][4];
#pragma unroll
                for (int h2 = 0; h2 < 2; h2++) { // 16 dims per ldmatrix.x4.trans: n-tiles 2nn, 2nn+1
                    const int nn = 2 * n4 + h2;
                    const uint32_t voff = key * 256 + (((2 * nn + v_cg) ^ (key & 7)) << 4);
                    ldsm4t(vh[h2], sVh + voff);
                    ldsm4t(vl[h2], sVl + voff);
                }
#pragma unroll
                for (int j = 0; j < 4; j++) mma_f16(o[4 * n4 + j], pl[0], pl[1], pl[2], pl[3], vh[j >> 1][2 * (j & 1)], vh[j >> 1][2 * (j & 1) + 1]);
#pragma unroll
                for (int j = 0; j < 4; j++) mma_f16(o[4 * n4 + j], ph[0], ph[1], ph[2], ph[3], vl[j >> 1][2 * (j & 1)], vl[j >> 1][2 * (j & 1) + 1]);
#pragma unroll
                for (int j = 0; j < 4; j++) mma_f16(o[4 * n4 + j], ph[0], ph[1], ph[2], ph[3], vh[j >> 1][2 * (j & 1)], vh[j >> 1][2 * (j & 1) + 1]);
            }
        }
        __syncthreads(); // everybody is done with stage `st` before the next iteration's loads overwrite it
    }
    // row sums live spread over the quad
    l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
    l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
    l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
    const float i0 = __fdiv_rn(1.0f, l0), i1 = __fdiv_rn(1.0f, l1);
    const int tq0 = q0 + r0 / KVMUL, tq1 = q0 + r1 / KVMUL;
    float *d0 = out + (size_t)tq0 * AH + (size_t)(kvhd * KVMUL + r0 % KVMUL) * HEAD_DIM + 2 * t;
    float *d1 = out + (size_t)tq1 * AH + (size_t)(kvhd * KVMUL + r1 % KVMUL) * HEAD_DIM + 2 * t;
#pragma unroll
    for (int n = 0; n < 16; n++) {
        if (tq0 < T) *reinterpret_cast<float2 *>(d0 + 8 * n) = make_float2(__fmul_rn(o[n][0], i0), __fmul_rn(o[n][1], i0));
        if (tq1 < T) *reinterpret_cast<float2 *>(d1 + 8 * n) = make_float2(__fmul_rn(o[n][2], i1), __fmul_rn(o[n][3], i1));
    }
}

// ------------------------------------------------------------------------------------------
// Batched prefill under tensor parallelism: the row-parallel GEMMs (o_proj, down_proj) leave a PARTIAL [T][dim] f32 block in
// this rank's part of the exchange buffer; after a cross-GPU barrier every rank adds the tp partials in RANK ORDER (so all
// ranks hold bit-identical residual streams, the same order as the decode path's exchange) over NVLink peer loads and folds
// them into its residual stream: T * dim * 4 bytes per sub-block and peer -- the bandwidth-bound exchange of SURVEY 8(e).
// Two partial buffers alternate (o_proj / down), so one barrier per exchange is enough: a buffer is rewritten only after
// the NEXT exchange's barrier, which a rank reaches after it has finished reading.
// ------------------------------------------------------------------------------------------
struct PfPeers {
    const float *part[MEGA_MAX_TP];        // every rank's partial block [Tcap][dim] (peer memory)
    unsigned long long *ctr[MEGA_MAX_TP];  // every rank's arrival counter (peer memory)
};
// one thread: tell every rank (this one included) that this rank's partial block is complete, wait until all tp ranks have said so
__global__ void k_pf_xbarrier(PfPeers p, int tp, int rank, unsigned long long target, int *status) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    __threadfence_system(); // the GEMM that wrote the block ran before this kernel on the same stream
    for (int r = 0; r < tp; r++) asm volatile("red.release.sys.global.add.u64 [%0], %1;" ::"l"(p.ctr[r]), "l"(1ULL) : "memory");
    const long long t0 = clock64();
    unsigned long long v;
    do {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p.ctr[rank]) : "memory");
        if (v < target && clock64() - t0 > 6000000000LL) { // ~3 s: a peer is gone; never hang the GPU
            atomicExch(status, 11);
            return;
        }
    } while (v < target);
}
// For tp > 2 the same sum as a reduce-scatter + all-gather over the same peer mappings (2 (tp-1)/tp blocks over NVLink per rank instead
// of tp-1): rank r sums slice r of all tp partial blocks in rank order and writes it back into ITS OWN block (nobody else reads that
// slice of it), a second barrier, then every rank adds slice r of rank r's block to its residual stream.  Same values as the direct form.
__global__ void __launch_bounds__(256) k_pf_reduce_scatter(PfPeers p, float *own, int tp, int rank, size_t n4) {
    const size_t lo = n4 * rank / tp, hi = n4 * (rank + 1) / tp;
    for (size_t i = lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (size_t)gridDim.x * blockDim.x) {
        float4 s = __ldcg(reinterpret_cast<const float4 *>(p.part[0]) + i);
        for (int r = 1; r < tp; r++) {
            const float4 v = __ldcg(reinterpret_cast<const float4 *>(p.part[r]) + i);
            s.x = __fadd_rn(s.x, v.x);
            s.y = __fadd_rn(s.y, v.y);
            s.z = __fadd_rn(s.z, v.z);
            s.w = __fadd_rn(s.w, v.w);
        }
        reinterpret_cast<float4 *>(own)[i] = s;
    }
}
// grid.y = owner rank of the slice
__global__ void __launch_bounds__(256) k_pf_allgather_resid(float *x, PfPeers p, int tp, size_t n4) {
    const int r = blockIdx.y;
    const size_t lo = n4 * r / tp, hi = n4 * (r + 1) / tp;
    for (size_t i = lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (size_t)gridDim.x * blockDim.x) {
        const float4 s = __ldcg(reinterpret_cast<const float4 *>(p.part[r]) + i);
        float4 o = reinterpret_cast<float4 *>(x)[i];
        o.x = __fadd_rn(o.x, s.x);
        o.y = __fadd_rn(o.y, s.y);
        o.z = __fadd_rn(o.z, s.z);
        o.w = __fadd_rn(o.w, s.w);
        reinterpret_cast<float4 *>(x)[i] = o;
    }
}
// x[t][c] += sum over ranks (in rank order) of part_r[t][c]      n4 = T * dim / 4
__global__ void __launch_bounds__(256) k_pf_allreduce_resid(float *x, PfPeers p, int tp, size_t n4) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        float4 s = __ldcg(reinterpret_cast<const float4 *>(p.part[0]) + i);
        for (int r = 1; r < tp; r++) {
            const float4 v = __ldcg(reinterpret_cast<const float4 *>(p.part[r]) + i);
            s.x = __fadd_rn(s.x, v.x);
            s.y = __fadd_rn(s.y, v.y);
            s.z = __fadd_rn(s.z, v.z);
            s.w = __fadd_rn(s.w, v.w);
        }
        float4 o = reinterpret_cast<float4 *>(x)[i];
        o.x = __fadd_rn(o.x, s.x);
        o.y = __fadd_rn(o.y, s.y);
        o.z = __fadd_rn(o.z, s.z);
        o.w = __fadd_rn(o.w, s.w);
        reinterpret_cast<float4 *>(x)[i] = o;
    }
}

// [rows][ng] -> [ng][rows] (weight scales, once at load)
__global__ void k_transpose_f32(const float *__restrict__ in, float *out, int rows, int cols) {
    __shared__ float tile[32][33];
    int c = blockIdx.x * 32 + threadIdx.x, r = blockIdx.y * 32 + threadIdx.y;
    for (int j = 0; j < 32; j += 8)
        if (r + j < rows && c < cols) tile[threadIdx.y + j][threadIdx.x] = in[(size_t)(r + j) * cols + c];
    __syncthreads();
    int oc = blockIdx.y * 32 + threadIdx.x, orow = blockIdx.x * 32 + threadIdx.y;
    for (int j = 0; j < 32; j += 8)
        if (orow + j < cols && oc < rows) out[(size_t)(orow + j) * rows + oc] = tile[threadIdx.x][threadIdx.y + j];
}

} // namespace q3
