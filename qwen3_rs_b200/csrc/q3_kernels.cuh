// q3_kernels.cuh -- hand-written sm_100a kernels for the qwen3-rs quantized decode path
// (multi-kernel variant; the persistent single-launch variant lives in q3_mega.cuh and reuses
// the device functions defined here).
//
// Arithmetic follows the reference op by op (file:line cited per kernel); floats are IEEE
// (no fast-math: true division, sqrtf, roundf, expf) and products/sums that the reference
// keeps separate are kept separate with __fmul_rn/__fadd_rn where contraction would change
// a quantisation input.  Only the ORDER of float reductions differs from the reference
// (parallel trees instead of left folds) -- see DESIGN.md "Numerics".
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace q3 {

constexpr int HEAD_DIM = 128;       // all Qwen3 models; enforced at load
constexpr float NORM_EPS = 1e-6f;   // layers.rs:6
constexpr int ATTN_MAX_SPLITS = 32; // split-K slots per kv head
constexpr int ATTN_MIN_CHUNK = 128; // positions per split before another split is opened

// ------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int4 ldg_stream(const int4 *p) {
    // weights are read exactly once per token: bypass L1
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
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
__device__ __forceinline__ int dot16(const int4 &w, const int4 &x, int acc) {
    acc = __dp4a(w.x, x.x, acc);
    acc = __dp4a(w.y, x.y, acc);
    acc = __dp4a(w.z, x.z, acc);
    acc = __dp4a(w.w, x.w, acc);
    return acc;
}
// Rust `f32 as i8` after f32::round (tensor.rs:116): round half away, saturate, NaN -> 0.
__device__ __forceinline__ int quant_one(float v, float scale) {
    float qv = (scale != 0.0f) ? __fdiv_rn(v, scale) : 0.0f;
    float r = roundf(qv);
    if (r != r) return 0;
    r = fminf(fmaxf(r, -128.0f), 127.0f);
    return (int)r;
}
__device__ __forceinline__ uint32_t pack4(int a, int b, int c, int d) {
    return (uint32_t)(a & 0xff) | ((uint32_t)(b & 0xff) << 8) | ((uint32_t)(c & 0xff) << 16) |
           ((uint32_t)(d & 0xff) << 24);
}
// f32::total_cmp key (sampler.rs:58): monotone signed integer image of the float.
__device__ __forceinline__ int total_key(float f) {
    int b = __float_as_int(f);
    return b ^ (int)(((unsigned)(b >> 31)) >> 1);
}

// ------------------------------------------------------------------------------------------
// Reference-order ("exact") mode.  The reference's floats come from glibc's libm; its expf
// (sysdeps/ieee754/flt-32/e_expf.c, glibc 2.27+; the algorithm of ARM optimized-routines) is
// a double-precision table + cubic evaluated in a fixed order, restated here so that
// exp() inside softmax / SwiGLU yields the same f32 bits on the device.  Table entries are
// 2^(i/32) as correctly rounded doubles minus (i << 47) (checked with 80-digit arithmetic).
// ------------------------------------------------------------------------------------------
__device__ __constant__ unsigned long long EXP2F_TAB[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull};

__device__ __forceinline__ float expf_ref(float x) {
    const unsigned abstop = (__float_as_uint(x) >> 20) & 0x7ff;
    if (abstop >= 0x42b) { // |x| >= 88 or nan
        if (__float_as_uint(x) == 0xff800000u) return 0.0f;
        if (abstop >= 0x7f8) return x + x;
        if (x > 0x1.62e42ep6f) return INFINITY;
        if (x < -0x1.9fe368p6f) return 0.0f;
    }
    // x86-64 glibc dispatches to its FMA build (__expf_fma, compiled with -mfma and GCC's default
    // -ffp-contract=fast) on every AVX2 host, so the products below are fused into the following
    // add exactly as that build does: kd = fma(InvLn2N, x, SHIFT), r = fma(InvLn2N, x, -kd), and
    // the three polynomial steps.  (Checked against glibc 2.39 on 4M+ inputs incl. hard cases.)
    const double xd = (double)x;
    const double InvLn2N = 0x1.71547652b82fep+0 * 32.0;
    const double SHIFT = 0x1.8p+52;
    double kd = __fma_rn(InvLn2N, xd, SHIFT);
    const unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
    kd = __dsub_rn(kd, SHIFT);
    const double r = __fma_rn(InvLn2N, xd, -kd);
    unsigned long long t = EXP2F_TAB[ki & 31];
    t += ki << (52 - 5);
    const double sc = __longlong_as_double((long long)t);
    const double C0 = 0x1.c6af84b912394p-5 / 32.0 / 32.0 / 32.0, C1 = 0x1.ebfce50fac4f3p-3 / 32.0 / 32.0,
                 C2 = 0x1.62e42ff0c52d6p-1 / 32.0;
    const double zz = __fma_rn(C0, r, C1);
    const double r2 = __dmul_rn(r, r);
    double y = __fma_rn(C2, r, 1.0);
    y = __fma_rn(zz, r2, y);
    y = __dmul_rn(y, sc);
    return (float)y;
}
template <bool ORDERED>
__device__ __forceinline__ float exp_sel(float x) {
    return ORDERED ? expf_ref(x) : expf(x);
}

// Quantise 4 consecutive values held by each of GS/4 adjacent lanes (one group = GS/4 lanes).
// tensor.rs:91-119: wmax = fold(0, max|x|), scale = wmax/127, q = round(x/scale).
//
// round(x/scale) without an IEEE division per element: t = x * rcp(scale) is within 2^-22 relative
// (< 4e-5 absolute, |t| <= 127) of the real quotient, and so is the correctly rounded quotient the
// reference computes; unless t lies within 2e-4 of a half-integer both round to the same integer
// (ties included: they are inside that window).  Elements inside the window (0.04 %) take the exact
// path.  NaN / zero-scale groups: t is NaN, cvt gives 0 -- what Rust's `NaN as i8` gives.
__device__ __forceinline__ int quant_fast(float v, float scale, float inv) {
    const float t = __fmul_rn(v, inv);
    const float n = rintf(t);
    if (!(fabsf(fabsf(t - n) - 0.5f) >= 2e-4f)) return quant_one(v, scale); // also taken when t is inf / NaN (denormal or zero scale)
    return __float2int_rn(n);
}
template <int GS>
__device__ __forceinline__ void quantize_group4(const float4 &y, uint32_t &packed, float &scale) {
    constexpr int LANES = GS / 4;
    static_assert(LANES >= 1 && LANES <= 32, "group size");
    float m = fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w)));
    m = fmaxf(m, 0.0f);
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    scale = __fdiv_rn(m, 127.0f);
    const float inv = __frcp_rn(scale);
    packed = pack4(quant_fast(y.x, scale, inv), quant_fast(y.y, scale, inv), quant_fast(y.z, scale, inv), quant_fast(y.w, scale, inv));
}

// ------------------------------------------------------------------------------------------
// RMSNorm (+ optional embedding gather) + group quantise.        one CTA, 1024 threads
//   layers.rs:72-76 (embedding row, dequantised on the fly: tensor.rs:72-80),
//   layers.rs:109-130 (RMSNorm), tensor.rs:91-119 (quantize).
// x_io: residual stream (read; written when gathering the embedding or when inplace_norm).
// ------------------------------------------------------------------------------------------
struct NormQuantArgs {
    float *x;              // [n] residual stream
    const float *w;        // [n] norm weight
    int8_t *q;             // [n]
    float *s;              // [n/GS]
    int n;
    const int8_t *embed_q; // non-null: x = dequant(embed row *token) first
    const float *embed_s;
    const int *token;
    int write_normed;      // 1: x <- normed value (final norm is in place, qwen3.rs:72)
};

// ORDERED: the sum of squares is the reference's left fold (one thread, element order), so the
// normalisation factor -- and with it every int8 activation -- is bit-identical to the reference.
template <int GS, bool ORDERED = false>
__global__ void __launch_bounds__(1024) k_rmsnorm_quant(NormQuantArgs a) {
    extern __shared__ __align__(16) float s_x[]; // ORDERED only: n floats
    __shared__ float red[32];
    __shared__ float s_f;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n4 = a.n >> 2;
    constexpr int MAXV = 4; // up to 16384 elements
    float4 v[MAXV];
    float ss = 0.0f;
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        int i4 = tid + k * 1024;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i4 < n4) {
            if (a.embed_q) {
                size_t base = (size_t)(*a.token) * a.n + (size_t)i4 * 4;
                char4 e = *reinterpret_cast<const char4 *>(a.embed_q + base);
                float sc = a.embed_s[base / GS];
                v[k] = make_float4((float)e.x * sc, (float)e.y * sc, (float)e.z * sc, (float)e.w * sc);
                reinterpret_cast<float4 *>(a.x)[i4] = v[k];
            } else {
                v[k] = reinterpret_cast<const float4 *>(a.x)[i4];
            }
            if (ORDERED) reinterpret_cast<float4 *>(s_x)[i4] = v[k];
            ss += __fmul_rn(v[k].x, v[k].x);
            ss += __fmul_rn(v[k].y, v[k].y);
            ss += __fmul_rn(v[k].z, v[k].z);
            ss += __fmul_rn(v[k].w, v[k].w);
        }
    }
    if (ORDERED) {
        __syncthreads();
        if (tid == 0) { // layers.rs:113: input.iter().map(|x| x*x).sum::<f32>()
            float t = 0.0f;
            for (int i = 0; i < a.n; i++) t = __fadd_rn(t, __fmul_rn(s_x[i], s_x[i]));
            s_f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(t, (float)a.n), NORM_EPS)));
        }
    } else {
        ss = warp_sum(ss);
        if (lane == 0) red[warp] = ss;
        __syncthreads();
        if (warp == 0) {
            float t = red[lane];
            t = warp_sum(t);
            if (lane == 0) s_f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(t, (float)a.n), NORM_EPS)));
        }
    }
    __syncthreads();
    const float f = s_f;
#pragma unroll
    for (int k = 0; k < MAXV; k++) {
        int i4 = tid + k * 1024;
        // whole warps are in or out together (n is a multiple of 128), so the shuffles are safe
        if (i4 - lane < n4) {
            float4 y = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i4 < n4) {
                float4 w = reinterpret_cast<const float4 *>(a.w)[i4];
                y.x = __fmul_rn(w.x, __fmul_rn(f, v[k].x));
                y.y = __fmul_rn(w.y, __fmul_rn(f, v[k].y));
                y.z = __fmul_rn(w.z, __fmul_rn(f, v[k].z));
                y.w = __fmul_rn(w.w, __fmul_rn(f, v[k].w));
            }
            uint32_t packed;
            float scale;
            quantize_group4<GS>(y, packed, scale);
            if (i4 < n4) {
                reinterpret_cast<uint32_t *>(a.q)[i4] = packed;
                if ((i4 % (GS / 4)) == 0) a.s[i4 / (GS / 4)] = scale;
                if (a.write_normed) reinterpret_cast<float4 *>(a.x)[i4] = y;
            }
        }
    }
}

// Plain RMSNorm (operator-level test entry; layers.rs:109-119).
__global__ void __launch_bounds__(1024) k_rmsnorm(const float *x, const float *w, float *out, int n) {
    __shared__ float red[32];
    __shared__ float s_f;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float ss = 0.0f;
    for (int i = tid; i < n; i += 1024) ss += __fmul_rn(x[i], x[i]);
    ss = warp_sum(ss);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    if (warp == 0) {
        float t = warp_sum(red[lane]);
        if (lane == 0) s_f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(t, (float)n), NORM_EPS)));
    }
    __syncthreads();
    const float f = s_f;
    for (int i = tid; i < n; i += 1024) out[i] = __fmul_rn(w[i], __fmul_rn(f, x[i]));
}

// ------------------------------------------------------------------------------------------
// Group quantise of an f32 vector (tensor.rs:91-119).   grid-stride, any n % GS == 0
// ------------------------------------------------------------------------------------------
template <int GS>
__global__ void __launch_bounds__(256) k_quantize(const float *__restrict__ x, int n, int8_t *q, float *s) {
    const int n4 = n >> 2;
    const int lane = threadIdx.x & 31;
    for (int base = (blockIdx.x * blockDim.x + threadIdx.x) - lane; base < n4; base += gridDim.x * blockDim.x) {
        int i4 = base + lane;
        float4 y = (i4 < n4) ? reinterpret_cast<const float4 *>(x)[i4] : make_float4(0.f, 0.f, 0.f, 0.f);
        uint32_t packed;
        float scale;
        quantize_group4<GS>(y, packed, scale);
        if (i4 < n4) {
            reinterpret_cast<uint32_t *>(q)[i4] = packed;
            if ((i4 % (GS / 4)) == 0) s[i4 / (GS / 4)] = scale;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Batch-1 int8 GEMV with per-group f32 scales (tensor.rs:23-62).
//   out[r] = sum_g ( (f32)(sum_k xq[g,k]*wq[r,g,k]) * ws[r,g] ) * xs[g]
// Row-major weights [rows][K] + scales [rows][K/GS].  256 threads = 8 warps; each warp owns a
// PAIR of rows per step (rows 2p, 2p+1) and streams them with 128-bit L1-bypassing loads;
// GS/16 adjacent lanes share one group, the int32 group dot is completed with shuffles and is
// exactly the reference's i32 sum.  x (int8 + scales) is staged once per CTA in shared memory.
// ------------------------------------------------------------------------------------------
enum GemvEpi { EPI_STORE = 0, EPI_QKV = 1, EPI_RESID = 2, EPI_SWIGLU = 3 };

struct GemvArgs {
    const int8_t *wq;
    const float *ws;
    const int8_t *xq;
    const float *xs;
    int K, rows;
    float *out;        // STORE: [rows]; RESID: x[rows] += ; SWIGLU: hb[rows/2]
    // QKV epilogue: rows [0,AH) -> q, [AH,AH+KV) -> kcache row, [AH+KV, AH+2KV) -> vcache row
    float *q;
    float *kc, *vc;    // layer base of the caches
    int AH, KV;
    const int *pos;
    int32_t *dots;     // optional [rows][K/GS] per-group integer dots (tests)
};

// ORDERED: the per-group f32 terms are parked in shared memory and folded left to right by one
// lane per row (tensor.rs:41-61 `.map(..).sum()`), making the row result bit-identical to the
// reference; EXPREF: exp() in the SwiGLU epilogue uses the glibc restatement.
template <int GS, int EPI, bool ORDERED = false, bool EXPREF = ORDERED>
__global__ void __launch_bounds__(256) k_gemv(GemvArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    int4 *sx = reinterpret_cast<int4 *>(smem);
    float *sxs = reinterpret_cast<float *>(smem + a.K);
    float *sterms = sxs + (a.K / GS) + (threadIdx.x >> 5) * 2 * (a.K / GS); // ORDERED: [warp][2][ng]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nchunk = a.K >> 4; // 16-byte chunks per row
    const int ng = a.K / GS;
    for (int i = tid; i < nchunk; i += 256) sx[i] = reinterpret_cast<const int4 *>(a.xq)[i];
    for (int i = tid; i < ng; i += 256) sxs[i] = a.xs[i];
    __syncthreads();

    constexpr int LPG = GS / 16; // lanes per group
    const int npairs = a.rows >> 1;
    for (int p = blockIdx.x * 8 + warp; p < npairs; p += gridDim.x * 8) {
        const size_t r0 = (size_t)(2 * p);
        const int4 *w0 = reinterpret_cast<const int4 *>(a.wq + r0 * a.K);
        const int4 *w1 = reinterpret_cast<const int4 *>(a.wq + (r0 + 1) * a.K);
        const float *s0 = a.ws + r0 * ng;
        const float *s1 = s0 + ng;
        float acc0 = 0.0f, acc1 = 0.0f;
        for (int c0 = 0; c0 < nchunk; c0 += 128) {
            int4 wa[4], wb[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                int c = c0 + u * 32 + lane;
                if (c < nchunk) {
                    wa[u] = ldg_stream(w0 + c);
                    wb[u] = ldg_stream(w1 + c);
                }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                int c = c0 + u * 32 + lane;
                bool ok = c < nchunk;
                int d0 = 0, d1 = 0;
                if (ok) {
                    int4 xv = sx[c];
                    d0 = dot16(wa[u], xv, 0);
                    d1 = dot16(wb[u], xv, 0);
                }
                if (c - lane < nchunk) { // warp-uniform: this step has at least one live lane
#pragma unroll
                    for (int o = LPG / 2; o > 0; o >>= 1) {
                        d0 += __shfl_xor_sync(0xffffffffu, d0, o);
                        d1 += __shfl_xor_sync(0xffffffffu, d1, o);
                    }
                    if (ok && (lane % LPG) == 0) {
                        int g = c / LPG;
                        float xsg = sxs[g];
                        // (dot as f32 * weight_scale) * input_scale   (tensor.rs:59)
                        float t0 = __fmul_rn(__fmul_rn((float)d0, __ldg(s0 + g)), xsg);
                        float t1 = __fmul_rn(__fmul_rn((float)d1, __ldg(s1 + g)), xsg);
                        if (ORDERED) {
                            sterms[g] = t0;
                            sterms[ng + g] = t1;
                        } else {
                            acc0 = __fadd_rn(acc0, t0);
                            acc1 = __fadd_rn(acc1, t1);
                        }
                        if (a.dots) {
                            a.dots[r0 * ng + g] = d0;
                            a.dots[(r0 + 1) * ng + g] = d1;
                        }
                    }
                }
            }
        }
        if (ORDERED) {
            __syncwarp();
            float t = 0.0f;
            if (lane < 2)
                for (int g = 0; g < ng; g++) t = __fadd_rn(t, sterms[lane * ng + g]);
            acc0 = __shfl_sync(0xffffffffu, t, 0);
            acc1 = __shfl_sync(0xffffffffu, t, 1);
            __syncwarp();
        } else {
            acc0 = warp_sum(acc0);
            acc1 = warp_sum(acc1);
        }
        if (lane == 0) {
            if (EPI == EPI_STORE) {
                a.out[r0] = acc0;
                a.out[r0 + 1] = acc1;
            } else if (EPI == EPI_RESID) { // ResidualConnection::forward, layers.rs:249-259
                a.out[r0] = __fadd_rn(a.out[r0], acc0);
                a.out[r0 + 1] = __fadd_rn(a.out[r0 + 1], acc1);
            } else if (EPI == EPI_SWIGLU) { // layers.rs:472-475: g * (1/(1+exp(-g))) * up
                float g = acc0;
                float sw = __fmul_rn(g, __fdiv_rn(1.0f, __fadd_rn(1.0f, exp_sel<EXPREF>(-g))));
                a.out[p] = __fmul_rn(sw, acc1);
            } else { // EPI_QKV, layers.rs:334-336: K and V go straight into the cache row of `pos`
                const int pos = *a.pos;
                int r = (int)r0;
                float *dst;
                if (r < a.AH) dst = a.q + r;
                else if (r < a.AH + a.KV) dst = a.kc + (size_t)pos * a.KV + (r - a.AH);
                else dst = a.vc + (size_t)pos * a.KV + (r - a.AH - a.KV);
                dst[0] = acc0;
                dst[1] = acc1;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// QK-RMSNorm + RoPE in place on q and on the freshly written K cache row.
//   layers.rs:346-372 (per head RMSNorm with the layer's [128] weight, then RoPE),
//   layers.rs:173-185 (half-split pairs (i, i+64)); cos/sin come from the host-computed table
//   (layers.rs:161-171 evaluated with glibc, bit-identical to the reference's libm calls).
// One warp per head; lane holds 4 consecutive dims; the pair partner lives in lane^16.
// ------------------------------------------------------------------------------------------
template <bool ORDERED = false>
__global__ void __launch_bounds__(128) k_qknorm_rope(float *q, float *kc_layer, const float *q_ln,
                                                     const float *k_ln, const float *rope, const int *pos_p,
                                                     int n_heads, int n_kv, int KV) {
    __shared__ float s_head[4][HEAD_DIM];
    const int lane = threadIdx.x & 31;
    const int head = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (head >= n_heads + n_kv) return;
    const int pos = *pos_p;
    float *p = head < n_heads ? q + (size_t)head * HEAD_DIM
                              : kc_layer + (size_t)pos * KV + (size_t)(head - n_heads) * HEAD_DIM;
    const float *w = head < n_heads ? q_ln : k_ln;
    float4 v = reinterpret_cast<float4 *>(p)[lane];
    float ss = __fmul_rn(v.x, v.x);
    ss = __fadd_rn(ss, __fmul_rn(v.y, v.y));
    ss = __fadd_rn(ss, __fmul_rn(v.z, v.z));
    ss = __fadd_rn(ss, __fmul_rn(v.w, v.w));
    if (ORDERED) { // left fold over the 128 dims in index order (layers.rs:113)
        float *sh = s_head[threadIdx.x >> 5];
        reinterpret_cast<float4 *>(sh)[lane] = v;
        __syncwarp();
        float t = 0.0f;
        if (lane == 0)
            for (int i = 0; i < HEAD_DIM; i++) t = __fadd_rn(t, __fmul_rn(sh[i], sh[i]));
        ss = __shfl_sync(0xffffffffu, t, 0);
    } else {
        ss = warp_sum(ss);
    }
    const float f = __fdiv_rn(1.0f, sqrtf(__fadd_rn(__fdiv_rn(ss, (float)HEAD_DIM), NORM_EPS)));
    float4 wv = reinterpret_cast<const float4 *>(w)[lane];
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
    // table row: [64][2] = (cos, sin) for pair index i; this lane covers i = 4*(lane&15)..+3
    const float4 *cs = reinterpret_cast<const float4 *>(rope + (size_t)pos * HEAD_DIM) + (lane & 15) * 2;
    float4 cs01 = cs[0], cs23 = cs[1]; // (c0,s0,c1,s1), (c2,s2,c3,s3)
    float4 r;
    if (lane < 16) { // first half: x*c - y*s
        r.x = __fsub_rn(__fmul_rn(y.x, cs01.x), __fmul_rn(o.x, cs01.y));
        r.y = __fsub_rn(__fmul_rn(y.y, cs01.z), __fmul_rn(o.y, cs01.w));
        r.z = __fsub_rn(__fmul_rn(y.z, cs23.x), __fmul_rn(o.z, cs23.y));
        r.w = __fsub_rn(__fmul_rn(y.w, cs23.z), __fmul_rn(o.w, cs23.w));
    } else { // second half: x*s + y*c, x = partner
        r.x = __fadd_rn(__fmul_rn(o.x, cs01.y), __fmul_rn(y.x, cs01.x));
        r.y = __fadd_rn(__fmul_rn(o.y, cs01.w), __fmul_rn(y.y, cs01.z));
        r.z = __fadd_rn(__fmul_rn(o.z, cs23.y), __fmul_rn(y.z, cs23.x));
        r.w = __fadd_rn(__fmul_rn(o.w, cs23.w), __fmul_rn(y.w, cs23.z));
    }
    reinterpret_cast<float4 *>(p)[lane] = r;
}

// ------------------------------------------------------------------------------------------
// GQA decode attention, split-K over the sequence (flash-decoding).
//   layers.rs:374-419: s_t = (q . k_t) / sqrt(128) for t in 0..=pos, softmax, out = sum a_t v_t.
// grid = (n_kv_heads, ATTN_MAX_SPLITS); the CTA streams its slice of K and V ONCE for all
// KVMUL query heads that share the kv head and leaves an un-normalised partial
// (m, l, acc[128]) per query head; k_attn_combine_quant merges the partials.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void attn_split_range(int pos, int split, int &t0, int &t1, int &nsplit) {
    int n = pos + 1;
    nsplit = (n + ATTN_MIN_CHUNK - 1) / ATTN_MIN_CHUNK;
    if (nsplit > ATTN_MAX_SPLITS) nsplit = ATTN_MAX_SPLITS;
    int per = (n + nsplit - 1) / nsplit;
    t0 = split * per;
    t1 = t0 + per;
    if (t1 > n) t1 = n;
}

constexpr int ATTN_PART_STRIDE = HEAD_DIM + 4; // acc[128], m, l, pad

template <int KVMUL>
__global__ void __launch_bounds__(128) k_attn_partial(const float *__restrict__ q, const float *__restrict__ kc,
                                                      const float *__restrict__ vc, float *part, const int *pos_p,
                                                      int KV, int n_heads) {
    const int kvh = blockIdx.x, split = blockIdx.y;
    const int pos = *pos_p;
    int t0, t1, nsplit;
    attn_split_range(pos, split, t0, t1, nsplit);
    if (split >= nsplit) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float scale = __fdiv_rn(1.0f, sqrtf((float)HEAD_DIM));
    float4 qv[KVMUL];
#pragma unroll
    for (int h = 0; h < KVMUL; h++)
        qv[h] = reinterpret_cast<const float4 *>(q + (size_t)(kvh * KVMUL + h) * HEAD_DIM)[lane];
    float m[KVMUL], l[KVMUL];
    float4 acc[KVMUL];
#pragma unroll
    for (int h = 0; h < KVMUL; h++) {
        m[h] = -INFINITY;
        l[h] = 0.0f;
        acc[h] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float *kbase = kc + (size_t)kvh * HEAD_DIM;
    const float *vbase = vc + (size_t)kvh * HEAD_DIM;
    for (int t = t0 + warp; t < t1; t += 4) {
        float4 kv = reinterpret_cast<const float4 *>(kbase + (size_t)t * KV)[lane];
        float4 vv = reinterpret_cast<const float4 *>(vbase + (size_t)t * KV)[lane];
        float s[KVMUL];
#pragma unroll
        for (int h = 0; h < KVMUL; h++)
            s[h] = qv[h].x * kv.x + qv[h].y * kv.y + qv[h].z * kv.z + qv[h].w * kv.w;
#pragma unroll
        for (int h = 0; h < KVMUL; h++) s[h] = __fmul_rn(warp_sum(s[h]), scale);
#pragma unroll
        for (int h = 0; h < KVMUL; h++) {
            float mn = fmaxf(m[h], s[h]);
            float corr = expf(m[h] - mn); // exp(-inf) = 0 on the first position
            float p = expf(s[h] - mn);
            l[h] = l[h] * corr + p;
            acc[h].x = acc[h].x * corr + p * vv.x;
            acc[h].y = acc[h].y * corr + p * vv.y;
            acc[h].z = acc[h].z * corr + p * vv.z;
            acc[h].w = acc[h].w * corr + p * vv.w;
            m[h] = mn;
        }
    }
    // merge the 4 warps
    __shared__ float sm_m[4][KVMUL], sm_l[4][KVMUL];
    __shared__ float4 sm_acc[4][KVMUL][32];
#pragma unroll
    for (int h = 0; h < KVMUL; h++) {
        if (lane == 0) {
            sm_m[warp][h] = m[h];
            sm_l[warp][h] = l[h];
        }
        sm_acc[warp][h][lane] = acc[h];
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int h = 0; h < KVMUL; h++) {
            float M = fmaxf(fmaxf(sm_m[0][h], sm_m[1][h]), fmaxf(sm_m[2][h], sm_m[3][h]));
            float L = 0.0f;
            float4 A = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int w = 0; w < 4; w++) {
                float mw = sm_m[w][h];
                float c = (mw == -INFINITY) ? 0.0f : expf(mw - M);
                L += sm_l[w][h] * c;
                float4 aw = sm_acc[w][h][lane];
                A.x += aw.x * c;
                A.y += aw.y * c;
                A.z += aw.z * c;
                A.w += aw.w * c;
            }
            float *dst = part + ((size_t)(kvh * KVMUL + h) * ATTN_MAX_SPLITS + split) * ATTN_PART_STRIDE;
            reinterpret_cast<float4 *>(dst)[lane] = A;
            if (lane == 0) {
                dst[HEAD_DIM] = M;
                dst[HEAD_DIM + 1] = L;
            }
        }
    }
}

// Merge split partials of one query head, normalise, and group-quantise the result
// (the quantize() before o_proj, qwen3.rs:152).  grid = n_heads, 128 threads (one per dim).
template <int GS>
__global__ void __launch_bounds__(128) k_attn_combine_quant(const float *__restrict__ part, const int *pos_p,
                                                            float *xb, int8_t *q, float *s) {
    const int head = blockIdx.x, d = threadIdx.x;
    const int pos = *pos_p;
    int t0, t1, nsplit;
    attn_split_range(pos, 0, t0, t1, nsplit);
    const float *base = part + (size_t)head * ATTN_MAX_SPLITS * ATTN_PART_STRIDE;
    float M = -INFINITY;
    for (int sidx = 0; sidx < nsplit; sidx++) M = fmaxf(M, base[sidx * ATTN_PART_STRIDE + HEAD_DIM]);
    float L = 0.0f, A = 0.0f;
    for (int sidx = 0; sidx < nsplit; sidx++) {
        const float *ps = base + sidx * ATTN_PART_STRIDE;
        float c = expf(ps[HEAD_DIM] - M);
        L += ps[HEAD_DIM + 1] * c;
        A += ps[d] * c;
    }
    float y = __fmul_rn(A, __fdiv_rn(1.0f, L)); // softmax multiplies by 1/sum (layers.rs:504-505)
    xb[head * HEAD_DIM + d] = y;
    // group quantise: HEAD_DIM/GS groups per head
    __shared__ int gmax[HEAD_DIM / 32];
    if (d < HEAD_DIM / 32) gmax[d] = 0;
    __syncthreads();
    constexpr int G = (GS > HEAD_DIM) ? HEAD_DIM : GS;
    atomicMax(&gmax[d / G], __float_as_int(fabsf(y)));
    __syncthreads();
    float scale = __fdiv_rn(__int_as_float(gmax[d / G]), 127.0f);
    q[head * HEAD_DIM + d] = (int8_t)quant_one(y, scale);
    if (d % G == 0) s[(head * HEAD_DIM + d) / G] = scale;
}

// Reference-order attention (exact mode): one CTA per query head, every reduction in the
// reference's order -- scores are left folds over the 128 dims (layers.rs:395-400), the softmax
// denominator a left fold over positions (layers.rs:497-503), the value mix a left fold over
// positions per output dim with separate multiply and add (layers.rs:408-417).  att: scratch
// [n_heads][seq_len] like the reference's `att` buffer.
__global__ void __launch_bounds__(128) k_attn_ordered(const float *__restrict__ q, const float *__restrict__ kc,
                                                      const float *__restrict__ vc, float *att, float *xb,
                                                      const int *pos_p, int KV, int kv_mul, int seq_len) {
    __shared__ float s_q[HEAD_DIM];
    __shared__ float red[4];
    __shared__ float s_bcast;
    const int head = blockIdx.x, tid = threadIdx.x;
    const int pos = *pos_p, n = pos + 1;
    const int kvh = head / kv_mul;
    float *a = att + (size_t)head * seq_len;
    s_q[tid] = q[(size_t)head * HEAD_DIM + tid];
    __syncthreads();
    const float scale = __fdiv_rn(1.0f, sqrtf((float)HEAD_DIM));
    float mx = -INFINITY;
    for (int t = tid; t < n; t += 128) {
        const float *k = kc + (size_t)t * KV + (size_t)kvh * HEAD_DIM;
        float sdot = 0.0f;
        for (int i = 0; i < HEAD_DIM; i++) sdot = __fadd_rn(sdot, __fmul_rn(s_q[i], k[i]));
        sdot = __fmul_rn(sdot, scale);
        a[t] = sdot;
        mx = fmaxf(mx, sdot);
    }
    mx = warp_max(mx);
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    for (int t = tid; t < n; t += 128) a[t] = expf_ref(__fsub_rn(a[t], mx));
    __syncthreads();
    if (tid == 0) {
        float sum = 0.0f;
        for (int t = 0; t < n; t++) sum = __fadd_rn(sum, a[t]);
        s_bcast = __fdiv_rn(1.0f, sum);
    }
    __syncthreads();
    const float inv = s_bcast;
    for (int t = tid; t < n; t += 128) a[t] = __fmul_rn(a[t], inv);
    __syncthreads();
    float o = 0.0f;
    const float *v = vc + (size_t)kvh * HEAD_DIM + tid;
    for (int t = 0; t < n; t++) o = __fadd_rn(o, __fmul_rn(a[t], v[(size_t)t * KV]));
    xb[(size_t)head * HEAD_DIM + tid] = o;
}

// ------------------------------------------------------------------------------------------
// Greedy argmax with the reference's tie rule (sampler.rs:57-59, max_by(total_cmp) keeps the
// LAST maximum).  One CTA; optionally feeds the token back and advances pos for on-device
// multi-step decode.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_argmax(const float *__restrict__ logits, int n, int *token_out,
                                                 int *token_feedback, int *pos_advance, int *history,
                                                 int *history_idx) {
    __shared__ long long red[32];
    long long best = (long long)0x8000000000000000LL;
    for (int i = threadIdx.x; i < n; i += 1024) {
        long long key = ((long long)total_key(logits[i]) << 32) | (unsigned)i; // ties -> larger index
        best = key > best ? key : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x < 32) {
        best = red[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other > best ? other : best;
        }
        if (threadIdx.x == 0) {
            int tok = (int)(best & 0xffffffffLL);
            *token_out = tok;
            if (token_feedback) *token_feedback = tok;
            if (pos_advance) *pos_advance += 1;
            if (history) {
                history[*history_idx] = tok;
                *history_idx += 1;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Per-row log-softmax at a target index + greedy argmax (q3_score, q3_op_logprobs).  One CTA per row of `logits`
// (row pitch ld floats), one streaming pass: each thread keeps the running max m (the value of its argmax key),
// sum s of expf(x - m) rescaled when m grows, and the key of its last maximum -- the total-order key of k_argmax, so
// the index is the reference's (sampler.rs:57-59: last index among equal maxima).  The per-thread partials are
// combined over a fixed shuffle / shared-memory tree, so the result depends on the row's values and LP_THREADS only:
// the same logits give the same bits however many rows are launched.  lp = (x[target] - m) - logf(s).
// ------------------------------------------------------------------------------------------
constexpr int LP_THREADS = 512;
constexpr int LP_BATCH = 8; // loads issued per thread before they are folded (in index order)

struct LpPart {
    long long key; // (total_key(max) << 32) | index
    float m, s;
};
// (a, b) -> a; commutative, so both lanes of a shuffle pair hold the same value
__device__ __forceinline__ void lp_combine(LpPart &a, const LpPart &b) {
    if (b.key > a.key) {
        a.s = b.s + (a.s == 0.0f ? 0.0f : a.s * expf(a.m - b.m));
        a.m = b.m;
        a.key = b.key;
    } else {
        a.s = a.s + (b.s == 0.0f ? 0.0f : b.s * expf(b.m - a.m));
    }
}
__device__ __forceinline__ LpPart lp_shfl(const LpPart &p, int o) {
    LpPart q;
    q.key = __shfl_xor_sync(0xffffffffu, p.key, o);
    q.m = __shfl_xor_sync(0xffffffffu, p.m, o);
    q.s = __shfl_xor_sync(0xffffffffu, p.s, o);
    return q;
}

// One thread's streaming pass over its elements x[tid], x[tid + LP_THREADS], ... of a row of n: the running max, the
// rescaled sum and the key of the last maximum.  each(i, v) sees every element the thread folds (k_topk_logprobs' histogram).
template <class F>
__device__ __forceinline__ void lp_accumulate(LpPart &p, const float *__restrict__ x, int n, int tid, F each) {
    p = LpPart{(long long)0x8000000000000000LL, -INFINITY, 0.0f};
    for (int base = tid; base < n; base += LP_BATCH * LP_THREADS) {
        float v[LP_BATCH];
#pragma unroll
        for (int k = 0; k < LP_BATCH; k++) {
            const int i = base + k * LP_THREADS;
            v[k] = i < n ? x[i] : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < LP_BATCH; k++) {
            const int i = base + k * LP_THREADS;
            if (i < n) {
                each(i, v[k]);
                const long long key = ((long long)total_key(v[k]) << 32) | (unsigned)i;
                if (key > p.key) { // new maximum (or an equal value at a later index: expf(0) = 1 either way)
                    p.s = (p.s == 0.0f ? 0.0f : p.s * expf(p.m - v[k])) + 1.0f;
                    p.m = v[k];
                    p.key = key;
                } else {
                    p.s += expf(v[k] - p.m);
                }
            }
        }
    }
}
__global__ void __launch_bounds__(LP_THREADS) k_logprobs(const float *__restrict__ logits, int n, size_t ld,
                                                         const int *__restrict__ targets, float *lp_out, int *argmax_out) {
    __shared__ LpPart red[LP_THREADS / 32];
    const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *x = logits + (size_t)row * ld;
    LpPart p;
    lp_accumulate(p, x, n, tid, [](int, float) {});
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lp_combine(p, lp_shfl(p, o));
    if (lane == 0) red[warp] = p;
    __syncthreads();
    if (warp == 0) {
        p = lane < LP_THREADS / 32 ? red[lane] : LpPart{(long long)0x8000000000000000LL, -INFINITY, 0.0f};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lp_combine(p, lp_shfl(p, o));
        if (lane == 0) {
            if (lp_out) lp_out[row] = __fsub_rn(__fsub_rn(x[targets[row]], p.m), logf(p.s));
            if (argmax_out) argmax_out[row] = (int)(p.key & 0xffffffffLL);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Per-row top-k log-probabilities (q3_score_topk, q3_op_topk_logprobs).  One CTA per row, k <= TOPK_MAX.  The k entries
// are the k largest 64-bit keys (total_key(x) << 32) | index -- descending value, ties to the larger index -- so ids[0] is
// k_logprobs' argmax and the selection is a function of the row alone.  lps[j] = (x[ids[j]] - m) - logf(s) with m, s from
// k_logprobs' own accumulation (lp_accumulate) and combine tree: at ids[j] == target it is q3_score's value bit for bit.
// Selection is a radix select on the key as an unsigned number, 11 bits per digit from the top:
//   1. the (m, s) pass also counts the top digit of every key into a shared histogram;
//   2. a scan finds the bin of the k-th largest key; all keys above that bin are in the top k;
//   3. if those keys plus the bin's hold at most TOPK_CAP, a second read gathers them and a bitonic sort orders them;
//   4. otherwise the next digit is counted over the bin's keys (another read of the row), down into the index bits.
// Keys are unique, so the bin of the last digit holds one key and the loop ends: an all-equal row takes 5 counting reads.
// ------------------------------------------------------------------------------------------
constexpr int TOPK_MAX = 64;
constexpr int TOPK_DIGIT = 11;                // bits per radix digit (the last one, bits 8..0, has 9)
constexpr int TOPK_BINS = 1 << TOPK_DIGIT;
constexpr int TOPK_CAP = 2048;                // candidates sorted in shared memory (16 KB)
static_assert(TOPK_BINS == 4 * LP_THREADS, "the bin scan gives each thread 4 bins");

// the key of k_argmax / k_logprobs as an unsigned number (same order)
__device__ __forceinline__ unsigned long long topk_key(float v, int i) {
    return ((unsigned long long)((unsigned)total_key(v) ^ 0x80000000u) << 32) | (unsigned)i;
}

__global__ void __launch_bounds__(LP_THREADS) k_topk_logprobs(const float *__restrict__ logits, int n, size_t ld, int k,
                                                              int *ids, float *lps, const int *__restrict__ targets,
                                                              float *lp_out, int *argmax_out) {
    __shared__ LpPart red[LP_THREADS / 32];
    __shared__ unsigned hist[TOPK_BINS];
    __shared__ unsigned long long cand[TOPK_CAP];
    __shared__ unsigned wsum[LP_THREADS / 32];
    __shared__ float s_m, s_s;
    __shared__ unsigned s_bin, s_gt, s_count;
    const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float *x = logits + (size_t)row * ld;
    for (int b = tid; b < TOPK_BINS; b += LP_THREADS) hist[b] = 0;
    if (tid == 0) s_count = 0;
    __syncthreads();
    LpPart p;
    lp_accumulate(p, x, n, tid, [&](int, float v) {
        atomicAdd(&hist[((unsigned)total_key(v) ^ 0x80000000u) >> (32 - TOPK_DIGIT)], 1u);
    });
    // k_logprobs' combine tree, step for step (its __syncthreads also completes the histogram)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lp_combine(p, lp_shfl(p, o));
    if (lane == 0) red[warp] = p;
    __syncthreads();
    if (warp == 0) {
        p = lane < LP_THREADS / 32 ? red[lane] : LpPart{(long long)0x8000000000000000LL, -INFINITY, 0.0f};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lp_combine(p, lp_shfl(p, o));
        if (lane == 0) {
            s_m = p.m;
            s_s = p.s;
            if (lp_out) lp_out[row] = __fsub_rn(__fsub_rn(x[targets[row]], p.m), logf(p.s));
            if (argmax_out) argmax_out[row] = (int)(p.key & 0xffffffffLL);
        }
    }
    unsigned long long sel = 0; // the key's digits chosen so far: every key in the top k is >= sel << shift
    int shift = 64;             // key bits below the chosen digits
    unsigned above = 0;         // keys above the chosen prefix: all in the top k
    unsigned need = (unsigned)k; // how many of the top k are still to be found under the chosen prefix
    for (;;) {
        const int width = shift >= TOPK_DIGIT ? TOPK_DIGIT : shift;
        // the bin holding the need-th largest key of this digit: each thread owns 4 bins, thread 0 the top ones
        unsigned h[4], c = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) c += h[j] = hist[TOPK_BINS - 1 - 4 * tid - j];
        unsigned incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) wsum[warp] = incl;
        __syncthreads();
        unsigned acc = incl - c;
        for (int w = 0; w < warp; w++) acc += wsum[w];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (acc < need && acc + h[j] >= need) {
                s_bin = TOPK_BINS - 1 - 4 * tid - j;
                s_gt = acc;
            }
            acc += h[j];
        }
        __syncthreads();
        const unsigned bin = s_bin, gt = s_gt;
        shift -= width;
        sel = (sel << width) | bin;
        above += gt;
        if (above + hist[bin] <= TOPK_CAP) break;
        need -= gt;
        // the next digit, counted over the keys under the chosen prefix (one more read of the row)
        const int nw = shift >= TOPK_DIGIT ? TOPK_DIGIT : shift;
        __syncthreads(); // every thread has read hist[bin]
        for (int b = tid; b < TOPK_BINS; b += LP_THREADS) hist[b] = 0;
        __syncthreads();
        for (int base = tid; base < n; base += LP_BATCH * LP_THREADS) {
            float v[LP_BATCH];
#pragma unroll
            for (int j = 0; j < LP_BATCH; j++) {
                const int i = base + j * LP_THREADS;
                v[j] = i < n ? x[i] : 0.0f;
            }
#pragma unroll
            for (int j = 0; j < LP_BATCH; j++) {
                const int i = base + j * LP_THREADS;
                const unsigned long long key = topk_key(v[j], i);
                if (i < n && (key >> shift) == sel) atomicAdd(&hist[(unsigned)(key >> (shift - nw)) & ((1u << nw) - 1)], 1u);
            }
        }
        __syncthreads();
    }
    // gather every key >= lo (above + hist[bin] of them, at least k) into shared memory, warp by warp
    const unsigned long long lo = sel << shift;
    for (int base0 = 0; base0 < n; base0 += LP_BATCH * LP_THREADS) { // uniform trip count: the ballots see full warps
        float v[LP_BATCH];
#pragma unroll
        for (int j = 0; j < LP_BATCH; j++) {
            const int i = base0 + tid + j * LP_THREADS;
            v[j] = i < n ? x[i] : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < LP_BATCH; j++) {
            const int i = base0 + tid + j * LP_THREADS;
            const unsigned long long key = topk_key(v[j], i);
            const bool take = i < n && key >= lo;
            const unsigned mask = __ballot_sync(0xffffffffu, take);
            if (mask) {
                unsigned off = 0;
                if (lane == 0) off = atomicAdd(&s_count, (unsigned)__popc(mask));
                off = __shfl_sync(0xffffffffu, off, 0) + __popc(mask & ((1u << lane) - 1));
                if (take && off < TOPK_CAP) cand[off] = key;
            }
        }
    }
    __syncthreads();
    const int cnt = (int)min(s_count, (unsigned)TOPK_CAP);
    int npad = 1;
    while (npad < cnt) npad <<= 1;
    for (int i = cnt + tid; i < npad; i += LP_THREADS) cand[i] = 0; // below every key that can be among the top k
    __syncthreads();
    // bitonic sort, descending
    for (int kk = 2; kk <= npad; kk <<= 1) {
        for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < npad; i += LP_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = cand[i], b = cand[ixj];
                    if ((a < b) == ((i & kk) == 0)) {
                        cand[i] = b;
                        cand[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    const float m = s_m, ls = logf(s_s);
    for (int j = tid; j < k; j += LP_THREADS) {
        const int id = (int)(cand[j] & 0xffffffffu);
        ids[(size_t)row * k + j] = id;
        lps[(size_t)row * k + j] = __fsub_rn(__fsub_rn(x[id], m), ls);
    }
}

// ------------------------------------------------------------------------------------------
// Exporter quantiser on the device (qwen3-export model_exporter.rs:104-161, SURVEY §8f-3):
// scale = max|w|/127 (1.0 for an all-zero group), q = clamp(rint(w/scale), -127, 127).
// rintf is round-half-to-even == round_half_to_even() (:321-338).
// ------------------------------------------------------------------------------------------
template <int GS>
__global__ void __launch_bounds__(256) k_quantize_q80(const float *__restrict__ w, size_t n, int8_t *q, float *s) {
    constexpr int LANES = GS / 4;
    const size_t n4 = n >> 2;
    const int lane = threadIdx.x & 31;
    for (size_t base = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) - lane; base < n4;
         base += (size_t)gridDim.x * blockDim.x) {
        size_t i4 = base + lane;
        float4 y = (i4 < n4) ? reinterpret_cast<const float4 *>(w)[i4] : make_float4(0.f, 0.f, 0.f, 0.f);
        float m = fmaxf(fmaxf(fabsf(y.x), fabsf(y.y)), fmaxf(fabsf(y.z), fabsf(y.w)));
        m = fmaxf(m, 0.0f);
#pragma unroll
        for (int o = LANES / 2; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float scale = m > 0.0f ? __fdiv_rn(m, 127.0f) : 1.0f;
        float v[4] = {y.x, y.y, y.z, y.w};
        int qi[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            int out = 0;
            if (scale > 0.0f) { // :130 (a denormal max can underflow the scale to 0)
                float r = rintf(__fdiv_rn(v[j], scale));
                // f32::clamp keeps NaN, `as i8` then maps it to 0 (:133)
                out = (r != r) ? 0 : (int)fminf(fmaxf(r, -127.0f), 127.0f);
            }
            qi[j] = out;
        }
        if (i4 < n4) {
            reinterpret_cast<uint32_t *>(q)[i4] = pack4(qi[0], qi[1], qi[2], qi[3]);
            if ((i4 % LANES) == 0) s[i4 / LANES] = scale;
        }
    }
}

} // namespace q3
