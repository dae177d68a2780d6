// kernels.cuh — hand-written sm_100a kernels for the VITS acoustic+vocoder forward pass.
//
// Data layout in HBM: every activation is TIME-MAJOR / channels-last fp32, `x[row][C]` with a
// row stride (ld) so that channel sub-ranges (coupling halves, gate halves) are plain pointer
// offsets.  A batch is PACKED along rows: utterance u owns rows
//     [off[u]*rate + u*extra, off[u+1]*rate + u*extra)
// where off[] is the token- or frame-offset table and `rate` the cumulative upsampling factor of
// the stage.  Every conv zero-pads at the edges of ITS OWN utterance (the reference never sees
// more than one utterance: batch is hard-wired to 1, multi_head_attention.cpp:208).
//
// Each kernel cites the reference function it replaces.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "rng.cuh"

namespace stts {

// ----------------------------------------------------------------------------------------------
// shared helpers
// ----------------------------------------------------------------------------------------------
struct Seg {
    const int* off;  // [B+1] base offsets (tokens or frames)
    int rate;        // rows per base unit
    int extra;       // extra rows per utterance (1 for the reflect-padded MS tail)
};
__device__ __forceinline__ int seg_start(const Seg& s, int u) { return s.off[u] * s.rate + u * s.extra; }
__device__ __forceinline__ int seg_len(const Seg& s, int u) { return (s.off[u + 1] - s.off[u]) * s.rate + s.extra; }

// nn_tanh, src/nn_op/nn_tanh.cpp:6-21: (e^x - e^-x)/(e^x + e^-x), inf -> 1e10, denominator floor 1e-8
__device__ __forceinline__ float tanh_ref(float x) {
    float a = expf(x), b = expf(-x);
    if (isinf(a)) a = 1e10f;
    if (isinf(b)) b = 1e10f;
    float d = a + b;
    if (d < 1e-8f) d = 1e-8f;
    return (a - b) / d;
}
// nn_sigmoid, src/nn_op/nn_sigmoid.cpp:3-7
__device__ __forceinline__ float sigmoid_ref(float x) { return 1.0f / (1.0f + expf(-x)); }
// nn_gelu, src/nn_op/nn_gelu.cpp:7-14
__device__ __forceinline__ float gelu_ref(float x) {
    float t = tanh_ref((x + x * x * x * 0.044715f) * 0.7978845608028654f);
    return (t + 1.0f) * x * 0.5f;
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
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// ----------------------------------------------------------------------------------------------
// K1. Conv1d as a tiled implicit GEMM on the CUDA cores (fp32 FFMA).
// Replaces nn_conv1d::forward (dense branch), src/nn_op/nn_conv1d.cpp:118-199, for every dense
// conv / 1x1 / (phase-expanded) ConvTranspose1d on the path, with the surrounding elementwise
// reference ops fused:
//   input  side: leaky-relu (nn_leaky_relu.cpp:6-27) applied while staging the tile
//   output side: bias (nn_conv1d.cpp:192-195), per-utterance speaker vector (WN.cpp:120-124,
//                Generator_hifigan.cpp:147-151, FixDurationPredictor.cpp:81-85), ReLU
//                (nn_relu.cpp), residual add (ResBlock1.cpp:65), MRF mean (Generator_MS.cpp:179-196),
//                WN gate tanh*sigmoid (WN.cpp:85-98), res/skip accumulation (WN.cpp:128-146),
//                coupling x1 -= m (ResidualCouplingLayer.cpp:58) via negated weights.
// GEMM orientation: M = time rows (BM per CTA), N = C_out (BN per CTA), K = C_in per tap.
// The x tile (BM + (k-1)*dil rows, 16 channels) is staged ONCE per channel chunk and reused by
// all k taps as row shifts; weight tiles [16][BN] stream through a cp.async double buffer.
// ----------------------------------------------------------------------------------------------
enum { ACT_NONE = 0, ACT_LEAKY = 1 };
enum { EPI_STORE = 0, EPI_RELU = 1, EPI_ACCUM = 2, EPI_ACCUM_DIV = 3, EPI_GATE = 4, EPI_RESSKIP = 5, EPI_TANH = 6 };

struct ConvP {
    const float* x; int ldx;
    const float* w; int CoutW;      // [k][Cin][CoutW], CoutW = round_up(Cout, 4)
    const float* bias;              // [Cout] or null
    float* y; int ldy;
    float* y2; int ldy2;            // EPI_RESSKIP: skip destination
    const float* res; int ldr;      // residual added before the epilogue mode (may alias y)
    const float* gvec; int ldg;     // per-utterance additive vector gvec[u*ldg + n] or null
    Seg seg;
    int Cin, Cout, k, dil, padl;
    int in_act; float in_slope;
    int epi; float div; int split; int y2_store;
};

template <int BM, int BN>
__global__ void __launch_bounds__((BM / 4) * (BN / 8)) conv_tile_kernel(const ConvP p) {
    constexpr int NT = (BM / 4) * (BN / 8), BK = 16, TXN = BN / 8;
    extern __shared__ __align__(16) float smem[];
    const int u = blockIdx.y;
    const int seg0 = seg_start(p.seg, u);
    const int len = seg_len(p.seg, u);
    const int t0 = blockIdx.x * BM;
    if (t0 >= len) return;
    const int n0 = blockIdx.z * BN;
    const int halo = (p.k - 1) * p.dil;
    const int XR = BM + halo;
    const int LDX = (XR + 4) & ~3;                 // multiple of 4 keeps ws 16B aligned
    float* xs = smem;                              // [BK][LDX]
    float* ws = smem + BK * LDX;                   // [2][BK][BN]
    const int tid = threadIdx.x;
    const int tx = tid % TXN, ty = tid / TXN;
    const bool xvec = ((p.ldx & 3) == 0) && ((((uintptr_t)p.x) & 15) == 0);

    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    const int nchunk = (p.Cin + BK - 1) / BK;
    for (int cc = 0; cc < nchunk; ++cc) {
        const int c0 = cc * BK;
        __syncthreads();  // previous chunk fully consumed before xs / ws are overwritten
        // ---- stage x tile, transposed to [c][row] -------------------------------------------
        for (int idx = tid; idx < XR * 4; idx += NT) {
            const int r = idx >> 2, q = idx & 3;
            const int tl = t0 + r - p.padl;
            const int c = c0 + q * 4;
            float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
            if (tl >= 0 && tl < len && c < p.Cin) {
                const float* src = p.x + (size_t)(seg0 + tl) * p.ldx + c;
                if (xvec && c + 3 < p.Cin) {
                    const float4 v = __ldg(reinterpret_cast<const float4*>(src));
                    v0 = v.x; v1 = v.y; v2 = v.z; v3 = v.w;
                } else {
                    v0 = __ldg(src);
                    if (c + 1 < p.Cin) v1 = __ldg(src + 1);
                    if (c + 2 < p.Cin) v2 = __ldg(src + 2);
                    if (c + 3 < p.Cin) v3 = __ldg(src + 3);
                }
                if (p.in_act == ACT_LEAKY) {
                    v0 = v0 < 0.f ? v0 * p.in_slope : v0;
                    v1 = v1 < 0.f ? v1 * p.in_slope : v1;
                    v2 = v2 < 0.f ? v2 * p.in_slope : v2;
                    v3 = v3 < 0.f ? v3 * p.in_slope : v3;
                }
            }
            xs[(q * 4 + 0) * LDX + r] = v0;
            xs[(q * 4 + 1) * LDX + r] = v1;
            xs[(q * 4 + 2) * LDX + r] = v2;
            xs[(q * 4 + 3) * LDX + r] = v3;
        }
        // ---- weight tile loader (cp.async, zero-fill out of range) ---------------------------
        auto load_w = [&](int tap, int buf) {
            float* dst = ws + buf * (BK * BN);
            for (int idx = tid; idx < BK * (BN / 4); idx += NT) {
                const int c = idx / (BN / 4), q = idx % (BN / 4);
                const int n = n0 + q * 4;
                float* d = dst + c * BN + q * 4;
                if (c0 + c < p.Cin && n < p.CoutW) {
                    cp_async16(d, p.w + ((size_t)tap * p.Cin + c0 + c) * p.CoutW + n);
                } else {
                    *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        };
        load_w(0, 0);
        cp_async_commit();
        for (int tap = 0; tap < p.k; ++tap) {
            if (tap + 1 < p.k) {
                load_w(tap + 1, (tap + 1) & 1);
                cp_async_commit();
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncthreads();
            const float* wb = ws + (tap & 1) * (BK * BN) + tx * 8;
            const float* xb = xs + ty * 4 + tap * p.dil;
#pragma unroll
            for (int c = 0; c < BK; ++c) {
                const float a0 = xb[c * LDX + 0], a1 = xb[c * LDX + 1], a2 = xb[c * LDX + 2], a3 = xb[c * LDX + 3];
                const float4 b0 = *reinterpret_cast<const float4*>(wb + c * BN);
                const float4 b1 = *reinterpret_cast<const float4*>(wb + c * BN + 4);
                const float a[4] = {a0, a1, a2, a3};
                const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
            }
            __syncthreads();
        }
    }

    // ---- epilogue --------------------------------------------------------------------------
    const int nb = n0 + tx * 8;
    float bv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int n = nb + j;
        float b = 0.f;
        if (n < p.Cout) {
            if (p.bias) b = __ldg(p.bias + n);
            if (p.gvec) b += __ldg(p.gvec + (size_t)u * p.ldg + n);
        }
        bv[j] = b;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int t = t0 + ty * 4 + i;
        if (t >= len) continue;
        const size_t row = (size_t)(seg0 + t);
        if (p.epi == EPI_GATE) {
            // channels are stored interleaved (tanh_j, sigmoid_j): WN.cpp:85-98
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                const int n = nb + j;
                if (n + 1 < p.Cout)
                    p.y[row * p.ldy + (n >> 1)] = tanh_ref(acc[i][j] + bv[j]) * sigmoid_ref(acc[i][j + 1] + bv[j + 1]);
            }
        } else if (p.epi == EPI_RESSKIP) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int n = nb + j;
                if (n >= p.Cout) continue;
                const float v = acc[i][j] + bv[j];
                if (n < p.split) {
                    float* d = p.y + row * p.ldy + n;      // x = x + res_acts        (WN.cpp:134)
                    *d = *d + v;
                } else {
                    float* d = p.y2 + row * p.ldy2 + (n - p.split);  // output += ... (WN.cpp:138,143)
                    *d = p.y2_store ? v : (*d + v);
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int n = nb + j;
                if (n >= p.Cout) continue;
                float v = acc[i][j] + bv[j];
                if (p.res) v = v + p.res[row * p.ldr + n];
                float* d = p.y + row * p.ldy + n;
                if (p.epi == EPI_RELU) v = v < 0.f ? 0.f : v;
                else if (p.epi == EPI_ACCUM) v = *d + v;
                else if (p.epi == EPI_ACCUM_DIV) v = (*d + v) / p.div;
                else if (p.epi == EPI_TANH) v = tanh_ref(v);
                *d = v;
            }
        }
    }
}

// ----------------------------------------------------------------------------------------------
// K2. Narrow conv (C_out <= 8): one thread per output row, weights in shared memory.
// Replaces nn_conv1d::forward for the 8- and 4-channel HiFi-GAN stages of multi_speakers.bin and
// conv_post (Generator_hifigan.cpp:176-180), where a 16-wide tensor/FFMA tile would be mostly padding.
// Same fused prologue/epilogue options as K1 (subset).
// ----------------------------------------------------------------------------------------------
template <int CO>
__global__ void __launch_bounds__(128) conv_narrow_kernel(const ConvP p) {
    extern __shared__ __align__(16) float wsm[];  // [k][Cin][CO]
    const int u = blockIdx.y;
    const int seg0 = seg_start(p.seg, u), len = seg_len(p.seg, u);
    const int t0 = blockIdx.x * blockDim.x;
    if (t0 >= len) return;
    for (int i = threadIdx.x; i < p.k * p.Cin * CO; i += blockDim.x) {
        const int n = i % CO, kc = i / CO;
        wsm[i] = n < p.Cout ? __ldg(p.w + (size_t)kc * p.CoutW + n) : 0.f;
    }
    __syncthreads();
    const int t = t0 + threadIdx.x;
    if (t >= len) return;
    float acc[CO];
#pragma unroll
    for (int n = 0; n < CO; ++n) acc[n] = 0.f;
    for (int tap = 0; tap < p.k; ++tap) {
        const int tl = t + tap * p.dil - p.padl;
        if (tl < 0 || tl >= len) continue;
        const float* xr = p.x + (size_t)(seg0 + tl) * p.ldx;
        const float* wr = wsm + tap * p.Cin * CO;
        for (int c = 0; c < p.Cin; ++c) {
            float xv = __ldg(xr + c);
            if (p.in_act == ACT_LEAKY) xv = xv < 0.f ? xv * p.in_slope : xv;
#pragma unroll
            for (int n = 0; n < CO; ++n) acc[n] = fmaf(xv, wr[c * CO + n], acc[n]);
        }
    }
    const size_t row = (size_t)(seg0 + t);
#pragma unroll
    for (int n = 0; n < CO; ++n) {
        if (n >= p.Cout) continue;
        float v = acc[n];
        if (p.bias) v += __ldg(p.bias + n);
        if (p.gvec) v += __ldg(p.gvec + (size_t)u * p.ldg + n);
        if (p.res) v = v + p.res[row * p.ldr + n];
        float* d = p.y + row * p.ldy + n;
        if (p.epi == EPI_RELU) v = v < 0.f ? 0.f : v;
        else if (p.epi == EPI_ACCUM) v = *d + v;
        else if (p.epi == EPI_ACCUM_DIV) v = (*d + v) / p.div;
        else if (p.epi == EPI_TANH) v = tanh_ref(v);
        *d = v;
    }
}

// ----------------------------------------------------------------------------------------------
// K3. Embedding gather * sqrt(hidden).  TextEncoder::forward, src/models/TextEncoder.cpp:57-63.
// emb is the file's column-major (vocab x embDim) table: e(v,c) = emb[c*vocab + v].
// ----------------------------------------------------------------------------------------------
__global__ void embed_kernel(const int* __restrict__ ids, const float* __restrict__ emb, float* __restrict__ x,
                             int ntok, int C, int vocab, float scale) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ntok * C) return;
    const int t = i / C, c = i % C;
    x[i] = __ldg(emb + (size_t)c * vocab + ids[t]) * scale;
}

// ----------------------------------------------------------------------------------------------
// K4. Relative-position multi-head attention (window w), flash-style, fp32.
// Replaces multi_head_attention::attention + helpers, src/modules/multi_head_attention.cpp:133-295:
//   s_ij = (q_i/sqrt(kc)).k_j + [|j-i|<=w] (q_i/sqrt(kc)).Ek[j-i+w]
//   p    = softmax_j(s)   (reference has no max-subtraction, nn_softmax.cpp:7; the online max used
//                          here is mathematically identical)
//   o_i  = sum_j p_ij v_j + sum_{|j-i|<=w} p_ij Ev[j-i+w]
// qkv: [rows][3*C] (q | k | v), one CTA = 16 queries of one head of one utterance, 4 warps.
// KC (channels per head) must be a multiple of 32 and <= 128.
// ----------------------------------------------------------------------------------------------
constexpr int RA_QPW = 8, RA_WARPS = 8, RA_THREADS = RA_WARPS * 32, RA_QT = RA_QPW * RA_WARPS;   // 64 queries per CTA
template <int KC>
__global__ void __launch_bounds__(RA_THREADS) relattn_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                       const float* __restrict__ embK, const float* __restrict__ embV,
                                                       Seg seg, int C, int win, int relRows) {
    constexpr int NL = KC / 32, KP = KC + 4, QT = RA_QT, QW = RA_QPW;   // KP % 4 == 0: float4 rows; 16*lane byte skew: conflict-free quarter-warps
    extern __shared__ __align__(16) float sm[];
    float* qs = sm;                    // [QT][KC]
    float* ks = qs + QT * KC;          // [32][KP]
    float* vs = ks + 32 * KP;          // [32][KP]
    float* ek = vs + 32 * KP;          // [R][KC]
    float* ev = ek + relRows * KC;     // [R][KC]
    float* rk = ev + relRows * KC;     // [QT][16] rel-k logits per query
    const int u = blockIdx.z, h = blockIdx.y;
    const int seg0 = seg_start(seg, u), len = seg_len(seg, u);
    const int q0 = blockIdx.x * QT;
    if (q0 >= len) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ld = 3 * C;
    const float inv = sqrtf((float)KC);
    const int R = 2 * win + 1;
    for (int i = tid; i < QT * KC; i += RA_THREADS) {
        const int r = i / KC, c = i % KC;
        const int t = q0 + r;
        qs[i] = t < len ? qkv[(size_t)(seg0 + t) * ld + h * KC + c] / inv : 0.f;
    }
    for (int i = tid; i < R * KC; i += RA_THREADS) {
        const int r = i / KC, c = i % KC;   // file is col-major (rows x cols): e(r,c) = p[c*rows + r]
        ek[i] = __ldg(embK + (size_t)c * relRows + r);
        ev[i] = __ldg(embV + (size_t)c * relRows + r);
    }
    __syncthreads();
    for (int i = tid; i < QT * R; i += RA_THREADS) {
        const int r = i / R, d = i % R;
        float s = 0.f;
        for (int c = 0; c < KC; ++c) s = fmaf(qs[r * KC + c], ek[d * KC + c], s);
        rk[r * 16 + d] = s;
    }
    // per-warp state for its QW queries (processed jointly: every K/V value read from smem feeds QW FMAs; a CTA of 64 queries
    // stages each K/V block once for 8 warps -- round 1 used 16 queries per CTA and re-staged K/V four times as often)
    float m[QW], l[QW], acc[QW][NL], sband[QW];
#pragma unroll
    for (int a = 0; a < QW; ++a) {
        m[a] = -INFINITY; l[a] = 0.f; sband[a] = -INFINITY;
#pragma unroll
        for (int c = 0; c < NL; ++c) acc[a][c] = 0.f;
    }
    const int qb = warp * QW;
    for (int j0 = 0; j0 < len; j0 += 32) {
        __syncthreads();
        for (int i = tid; i < 32 * (KC / 4); i += RA_THREADS) {
            const int r = i / (KC / 4), c4 = (i % (KC / 4)) * 4;
            const int t = j0 + r;
            float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
            if (t < len) {
                const float* src = qkv + (size_t)(seg0 + t) * ld + h * KC + c4;
                kv = *reinterpret_cast<const float4*>(src + C);
                vv = *reinterpret_cast<const float4*>(src + 2 * C);
            }
            *reinterpret_cast<float4*>(ks + r * KP + c4) = kv;
            *reinterpret_cast<float4*>(vs + r * KP + c4) = vv;
        }
        __syncthreads();
        const int j = j0 + lane;
        float s[QW];
#pragma unroll
        for (int a = 0; a < QW; ++a) s[a] = 0.f;
#pragma unroll 4
        for (int c = 0; c < KC; c += 4) {
            const float4 kv = *reinterpret_cast<const float4*>(ks + lane * KP + c);
#pragma unroll
            for (int a = 0; a < QW; ++a) {
                const float4 qv = *reinterpret_cast<const float4*>(qs + (qb + a) * KC + c);   // broadcast
                s[a] = fmaf(qv.x, kv.x, s[a]); s[a] = fmaf(qv.y, kv.y, s[a]);
                s[a] = fmaf(qv.z, kv.z, s[a]); s[a] = fmaf(qv.w, kv.w, s[a]);
            }
        }
        float pj[QW];
#pragma unroll
        for (int a = 0; a < QW; ++a) {
            const int i = q0 + qb + a;
            const int d = j - i + win;
            if (d >= 0 && d < R) s[a] += rk[(qb + a) * 16 + d];
            if (j >= len) s[a] = -INFINITY;
            {   // lane r keeps the raw score of relative offset r (key j = i + r - win)
                const int jr = i + lane - win;
                const int srcl = jr - j0;
                const float got = __shfl_sync(0xffffffffu, s[a], srcl & 31);
                if (lane < R && srcl >= 0 && srcl < 32 && jr >= 0 && jr < len && i < len) sband[a] = got;
            }
            const float cm = warp_max(s[a]);
            const float mn = fmaxf(m[a], cm);
            const float sc = expf(m[a] - mn);
            pj[a] = (j < len) ? expf(s[a] - mn) : 0.f;
            l[a] = l[a] * sc + warp_sum(pj[a]);
            m[a] = mn;
#pragma unroll
            for (int c = 0; c < NL; ++c) acc[a][c] *= sc;
        }
#pragma unroll 4
        for (int jj = 0; jj < 32; ++jj) {
            float v[NL];
#pragma unroll
            for (int c = 0; c < NL; ++c) v[c] = vs[jj * KP + lane + 32 * c];
#pragma unroll
            for (int a = 0; a < QW; ++a) {
                const float pb = __shfl_sync(0xffffffffu, pj[a], jj);
#pragma unroll
                for (int c = 0; c < NL; ++c) acc[a][c] = fmaf(pb, v[c], acc[a][c]);
            }
        }
    }
#pragma unroll
    for (int a = 0; a < QW; ++a) {
        const int qi = qb + a;
        const int i = q0 + qi;
        if (i >= len) continue;   // warp-uniform
        // normalised band probabilities -> rel-v term
        float pb = 0.f;
        if (lane < R && sband[a] != -INFINITY) pb = expf(sband[a] - m[a]) / l[a];
        float o[NL];
#pragma unroll
        for (int c = 0; c < NL; ++c) o[c] = acc[a][c] / l[a];
        for (int r = 0; r < R; ++r) {
            const float pr = __shfl_sync(0xffffffffu, pb, r);
#pragma unroll
            for (int c = 0; c < NL; ++c) o[c] = fmaf(pr, ev[r * KC + lane + 32 * c], o[c]);
        }
#pragma unroll
        for (int c = 0; c < NL; ++c) out[(size_t)(seg0 + i) * C + h * KC + lane + 32 * c] = o[c];
    }
}

// ----------------------------------------------------------------------------------------------
// K5. (a [+ b]) -> LayerNorm [-> GELU], one warp per row.
// Replaces nn_layer_norm::forward, src/nn_op/nn_layer_norm.cpp:65-86 (variance as E[x^2]-mean^2,
// eps 1e-5) fused with the residual add of attention_encoder.cpp:86-90 and with nn_gelu
// (DDSConv.cpp:100-105).  C <= 1024.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) add_ln_kernel(const float* a, const float* b,
                                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                                      float* y, int rows, int C, int gelu) {
    const int row = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    float v[32];
    float s = 0.f, sq = 0.f;
    const int n = (C + 31) / 32;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        if (i >= n) break;
        const int c = lane + 32 * i;
        float t = 0.f;
        if (c < C) {
            t = a[(size_t)row * C + c];
            if (b) t = t + b[(size_t)row * C + c];
        }
        v[i] = t;
        s += t;
        sq = fmaf(t, t, sq);
    }
    s = warp_sum(s);
    sq = warp_sum(sq);
    const float mean = s / (float)C;
    const float var = sq * (1.0f / (float)C) - mean * mean;
    const float den = sqrtf(var + 1e-5f);
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        if (i >= n) break;
        const int c = lane + 32 * i;
        if (c < C) {
            float o = ((v[i] - mean) / den) * __ldg(gamma + c) + __ldg(beta + c);
            if (gelu) o = gelu_ref(o);
            y[(size_t)row * C + c] = o;
        }
    }
}

// ----------------------------------------------------------------------------------------------
// K6. Depthwise conv (DDSConv's convs_sep).  nn_conv1d::forward `sep_` branch,
// src/nn_op/nn_conv1d.cpp:167-179; optional per-row add of `g` before (DDSConv.cpp:90-93 is applied
// by the caller once).  w: [k][C].
// ----------------------------------------------------------------------------------------------
__global__ void dwconv_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                              float* __restrict__ y, Seg seg, int C, int k, int dil, int pad) {
    const int u = blockIdx.y;
    const int seg0 = seg_start(seg, u), len = seg_len(seg, u);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= len * C) return;
    const int t = i / C, c = i % C;
    float acc = 0.f;
    for (int kk = 0; kk < k; ++kk) {
        const int tl = t + kk * dil - pad;
        if (tl >= 0 && tl < len) acc = fmaf(x[(size_t)(seg0 + tl) * C + c], __ldg(w + kk * C + c), acc);
    }
    if (bias) acc += __ldg(bias + c);
    y[(size_t)(seg0 + t) * C + c] = acc;
}

// y[r][c] = a[r][c] + b[r][c]   (DDSConv.cpp:107 `xx = xx + y`, :90-93 `xx = x + g`)
__global__ void add_kernel(const float* a, const float* b, float* y, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = a[i] + b[i];
}

// y[row][c] = x[row][c] + g[u][c]  (speaker vector broadcast over time, FixDurationPredictor.cpp:81-85)
__global__ void add_rowvec_kernel(const float* __restrict__ x, const float* __restrict__ g, int ldg,
                                  float* __restrict__ y, Seg seg, int C) {
    const int u = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= seg_len(seg, u) * C) return;
    const size_t o = (size_t)seg_start(seg, u) * C + i;
    y[o] = x[o] + __ldg(g + (size_t)u * ldg + (i % C));
}

// h[t][c] = x0[t]*w[c] + b[c]  — ConvFlow's 1->C `pre` conv (ConvFlow.cpp:247)
__global__ void expand1_kernel(const float* __restrict__ x0, const float* __restrict__ w, const float* __restrict__ b,
                               float* __restrict__ h, int rows, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * C) return;
    const int t = i / C, c = i % C;
    h[i] = fmaf(x0[t], __ldg(w + c), b ? __ldg(b + c) : 0.f);
}

// ----------------------------------------------------------------------------------------------
// K7. Inverse rational-quadratic spline (10 bins, tails +-5).
// Replaces unconstrained_rational_quadratic_spline + searchsorted, src/modules/ConvFlow.cpp:57-240,
// and the /sqrt(filter_channels) scaling of ConvFlow::forward :252-259.  One thread per token.
// h: [rows][ldh] with 10 widths | 10 heights | 9 derivatives.
// ----------------------------------------------------------------------------------------------
__global__ void rq_spline_inv_kernel(const float* __restrict__ h, int ldh, const float* x1,
                                     float* y1, int rows, float fsqrt) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows) return;
    constexpr int NB = 10;
    const float tail = 5.0f, MINW = 1e-3f, MINH = 1e-3f, MIND = 1e-3f;
    const float x = x1[t];
    const bool inside = (x < tail) && (x > -tail);
    if (!inside) { y1[t] = x; return; }
    const float* hr = h + (size_t)t * ldh;
    float wd[NB], ht[NB], dv[NB + 1];
    float sw = 0.f, sh = 0.f;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        wd[i] = expf(hr[i] / fsqrt);           // nn_softmax: exp / sum, no max subtraction
        ht[i] = expf(hr[NB + i] / fsqrt);
        sw += wd[i];
        sh += ht[i];
    }
    dv[0] = logf(expf(0.5397424172369522f) + 1.0f) + MIND;   // padded constant (ConvFlow.cpp:94-97)
    dv[NB] = dv[0];
#pragma unroll
    for (int i = 1; i < NB; ++i) dv[i] = logf(expf(hr[2 * NB + i - 1]) + 1.0f) + MIND;  // nn_softplus
    float cw[NB + 1], ch[NB + 1];
    float aw = 0.f, ah = 0.f;
    cw[0] = -tail; ch[0] = -tail;
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        const float wi = (wd[i] / sw) * (1.0f - MINW * NB) + MINW;
        const float hi = (ht[i] / sh) * (1.0f - MINH * NB) + MINH;
        aw += wi; ah += hi;                                    // nn_cumsum
        cw[i + 1] = aw * (2.0f * tail) + (-tail);
        ch[i + 1] = ah * (2.0f * tail) + (-tail);
    }
    cw[NB] = tail; ch[NB] = tail;
    int idx = -1;                                              // searchsorted over cumheights (+1e-6 on last)
#pragma unroll
    for (int i = 0; i <= NB; ++i) {
        const float loc = (i == NB) ? ch[i] + 1e-6f : ch[i];
        if (x >= loc) idx++;
    }
    idx = idx < 0 ? 0 : (idx > NB - 1 ? NB - 1 : idx);
    float icw = 0, ibw = 0, ich = 0, ih = 0, d0 = 0, d1 = 0;
#pragma unroll
    for (int i = 0; i < NB; ++i)
        if (i == idx) { icw = cw[i]; ibw = cw[i + 1] - cw[i]; ich = ch[i]; ih = ch[i + 1] - ch[i]; d0 = dv[i]; d1 = dv[i + 1]; }
    const float delta = ih / ibw;
    const float xm = x - ich;
    const float a = xm * (d0 + d1 - delta * 2.0f) + ih * (delta - d0);
    const float b = ih * d0 - xm * (d0 + d1 - 2.0f * delta);
    const float c = -(delta * xm);
    const float disc = b * b - a * c * 4.0f;
    const float root = (c * 2.0f) / (-b - sqrtf(disc));
    y1[t] = root * ibw + icw;
}

// logw = (a - m0) * exp(-logs0): ElementwiseAffine::forward, src/modules/ElementwiseAffine.cpp:44-58
__global__ void ea_kernel(const float* __restrict__ a, float* __restrict__ logw, int rows, float m0, float logs0) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < rows) logw[t] = (a[t] - m0) * expf(-logs0);
}

// ----------------------------------------------------------------------------------------------
// K8. Durations: w_ceil = ceil(exp(logw)*lengthScale) (or the forced value), per-utterance
// exclusive prefix (token -> first frame) and frame count = max(sum, 1).
// Replaces SynthesizerTrn.cpp:376-378 + the counting half of expandM :304-309.  One CTA per utterance.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) durations_kernel(const float* __restrict__ logw, int ldlogw,
                                                         const float* __restrict__ forced,
                                                         const float* __restrict__ lscale, const int* __restrict__ toff,
                                                         float* __restrict__ w_ceil, int* __restrict__ tok_first,
                                                         int* __restrict__ nframes) {
    __shared__ int part[256];
    __shared__ int carry;
    const int u = blockIdx.x;
    const int t0 = toff[u], n = toff[u + 1] - t0;
    const float ls = lscale[u];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 256) {
        const int i = base + threadIdx.x;
        int w = 0;
        if (i < n) {
            float wc;
            if (forced) wc = forced[t0 + i];
            else wc = ceilf(expf(logw[(size_t)(t0 + i) * ldlogw]) * ls);
            w_ceil[t0 + i] = wc;
            // NaN / inf / huge values (a cast of those is undefined) are clamped: at most 65536 frames per token; the host
            // rejects implausible totals before it plans the frame-level workspace
            w = (wc >= 0.f && wc <= 65536.f) ? (int)wc : (wc > 65536.f ? 65536 : 0);
        }
        part[threadIdx.x] = w;
        __syncthreads();
        for (int o = 1; o < 256; o <<= 1) {  // Hillis-Steele inclusive scan
            int v = threadIdx.x >= o ? part[threadIdx.x - o] : 0;
            __syncthreads();
            part[threadIdx.x] += v;
            __syncthreads();
        }
        if (i < n) tok_first[t0 + i] = carry + part[threadIdx.x] - w;
        __syncthreads();
        if (threadIdx.x == 255) carry += part[255];
        __syncthreads();
    }
    if (threadIdx.x == 0) nframes[u] = carry < 1 ? 1 : carry;   // nn_clamp_min(sum, 1.0)
}

// ----------------------------------------------------------------------------------------------
// K9. Length regulator: z_p[f] = m[token(f)]  (row repeat).  expandM, SynthesizerTrn.cpp:304-321,
// and z_p = m_expand (+ randn*exp(logs)*0), :383 — the RNG term is multiplied by noiseScale == 0
// (:357) and is not generated.  (regulate_noise_kernel below generates it for batches that sample.)
// ----------------------------------------------------------------------------------------------
// last token of utterance [t0, t0+n) whose first frame <= f, and whether f lies inside it (false on the padding frame of
// an all-zero-duration utterance)
__device__ __forceinline__ int regulate_token(const int* __restrict__ tok_first, const float* __restrict__ w_ceil, int t0, int n,
                                              int f, bool& valid) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (tok_first[t0 + mid] <= f) lo = mid; else hi = mid - 1;
    }
    valid = f < tok_first[t0 + lo] + (int)w_ceil[t0 + lo];
    return lo;
}

__global__ void regulate_kernel(const float* __restrict__ m, int ldm, const int* __restrict__ tok_first,
                                const float* __restrict__ w_ceil, const int* __restrict__ toff,
                                const int* __restrict__ foff, float* __restrict__ zp, int C) {
    const int u = blockIdx.y;
    const int f = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int F = foff[u + 1] - foff[u];
    if (f >= F) return;
    const int t0 = toff[u], n = toff[u + 1] - t0;
    bool valid;
    const int lo = regulate_token(tok_first, w_ceil, t0, n, f, valid);
    float* dst = zp + (size_t)(foff[u] + f) * C;
    const float* src = m + (size_t)(t0 + lo) * ldm;
    for (int c = lane; c < C; c += 32) dst[c] = valid ? src[c] : 0.f;
}

// K9s. Length regulator with the prior sampled (VITS SynthesizerTrn.infer): z_p = m + eps * exp(logs) * noise_scale, on the
// per-frame m / logs rows of expandM (both 0 on a padding frame, so z_p = eps * noise_scale there).  Same grid as
// regulate_kernel (one warp per frame); each lane draws one Philox call per channel quad q (counter (f, q, 0, 0), key = the
// utterance's seed, rng.cuh) and applies exp(logs) in registers, so no eps tensor exists in HBM.  An utterance with
// noise_scale == 0 copies m exactly as regulate_kernel does: the noise term is skipped, not multiplied (inf * 0 = NaN).
__global__ void __launch_bounds__(128) regulate_noise_kernel(const float* __restrict__ m, const float* __restrict__ logs, int ldm,
                                                             const int* __restrict__ tok_first, const float* __restrict__ w_ceil,
                                                             const int* __restrict__ toff, const int* __restrict__ foff,
                                                             float* __restrict__ zp, int C, const float* __restrict__ noise_scale,
                                                             const unsigned long long* __restrict__ seed) {
    const int u = blockIdx.y;
    const int f = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    const int F = foff[u + 1] - foff[u];
    if (f >= F) return;
    const int t0 = toff[u], n = toff[u + 1] - t0;
    bool valid;
    const int lo = regulate_token(tok_first, w_ceil, t0, n, f, valid);
    float* dst = zp + (size_t)(foff[u] + f) * C;
    const float* src = m + (size_t)(t0 + lo) * ldm;
    const float ns = noise_scale[u];
    if (ns == 0.f) {
        for (int c = lane; c < C; c += 32) dst[c] = valid ? src[c] : 0.f;
        return;
    }
    const float* ls = logs + (size_t)(t0 + lo) * ldm;
    const uint64_t key = seed[u];
    for (int q = lane; 4 * q < C; q += 32) {
        float e[4];
        philox_normals4((uint32_t)f, (uint32_t)q, 0u, 0u, key, e);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = 4 * q + j;
            if (c < C) dst[c] = valid ? src[c] + e[j] * expf(ls[c]) * ns : e[j] * ns;
        }
    }
}

// K9d. Initial rows of the stochastic duration predictor with noise (VITS: z = randn(2, T) * noise_scale_w, then nn_flip(z, 0),
// StochasticDurationPredictor.cpp:117-149): eps_r(t) from counter (t, 0, 1, 0) of the utterance's seed.  The flip swaps the two
// rows, so row 0 of the flipped z (`a`) is eps_1 * noise_scale_w and row 1 (`b`) is eps_0 * noise_scale_w.  noise_scale_w == 0
// writes exact zeros.  Grid (ceil(maxT / 128), B).
__global__ void __launch_bounds__(128) sdp_noise_kernel(float* __restrict__ a, float* __restrict__ b, const int* __restrict__ toff,
                                                        const float* __restrict__ noise_scale_w,
                                                        const unsigned long long* __restrict__ seed) {
    const int u = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int t0 = toff[u];
    if (t >= toff[u + 1] - t0) return;
    const float s = noise_scale_w[u];
    float e[4] = {0.f, 0.f, 0.f, 0.f};
    if (s != 0.f) philox_normals4((uint32_t)t, 0u, 1u, 0u, seed[u], e);
    a[t0 + t] = s != 0.f ? e[1] * s : 0.f;
    b[t0 + t] = s != 0.f ? e[0] * s : 0.f;
}

// gather speaker embedding rows: G[u][c] = emg(sid_u, c); emg col-major (spk x gin). SynthesizerTrn.cpp:363-372
__global__ void spk_gather_kernel(const float* __restrict__ emg, const int* __restrict__ sids, float* __restrict__ G,
                                  int B, int gin, int spk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * gin) return;
    const int u = i / gin, c = i % gin;
    int s = sids[u];
    if (s < 0 || s >= spk) s = 0;
    G[i] = __ldg(emg + (size_t)c * spk + s);
}

// reverse channel order of every row (only needed when the flow has an odd number of layers)
__global__ void chan_reverse_kernel(float* __restrict__ z, size_t rows, int C) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * (size_t)(C / 2)) return;
    const size_t r = i / (C / 2);
    const int c = (int)(i % (C / 2));
    float* p = z + r * C;
    const float a = p[c], b = p[C - 1 - c];
    p[c] = b; p[C - 1 - c] = a;
}

// ----------------------------------------------------------------------------------------------
// MS / iSTFT tail.
// K10. leaky(0.01) + reflect-pad(1,0): Generator_MS.cpp:198-206.  out rows per utterance = len+1.
// ----------------------------------------------------------------------------------------------
__global__ void refpad_leaky_kernel(const float* __restrict__ x, float* __restrict__ y, Seg sin, Seg sout, int C,
                                    float slope) {
    const int u = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int lin = seg_len(sin, u), lout = seg_len(sout, u);
    if (i >= lout * C) return;
    const int r = i / C, c = i % C;
    float v = 0.f;
    if (r == 0) { if (lin > 1) v = x[(size_t)(seg_start(sin, u) + 1) * C + c]; }
    else v = x[(size_t)(seg_start(sin, u) + r - 1) * C + c];
    v = v < 0.f ? v * slope : v;
    y[(size_t)(seg_start(sout, u) + r) * C + c] = v;
}

__constant__ float c_hann[16] = {0.0f, 0.03806023f, 0.14644661f, 0.30865828f, 0.5f, 0.69134172f, 0.85355339f,
                                 0.96193977f, 1.0f, 0.96193977f, 0.85355339f, 0.69134172f, 0.5f, 0.30865828f,
                                 0.14644661f, 0.03806023f};           // hann.cpp:3-5
__constant__ float c_hann_pow[16] = {0.0f, 0.00144858f, 0.02144661f, 0.09526994f, 0.25f, 0.47795337f, 0.72855339f,
                                     0.92532811f, 1.0f, 0.92532811f, 0.72855339f, 0.47795337f, 0.25f, 0.09526994f,
                                     0.02144661f, 0.00144858f};      // hann.cpp:6-9
__constant__ float c_cos16[16];  // cos(2*pi*m/16), filled at engine creation
__constant__ float c_sin16[16];

// K11. exp / pi*sin + 16-point real inverse DFT + Hann window, per (row, band).
// Replaces Generator_MS.cpp:210-221 and the per-frame half of iStft::forward, src/modules/iStft.cpp:63-105
// (kissfft real inverse uses only Re of DC and Nyquist, ei_kissfft_impl.h:376-405; scale 1/16).
// s: [rows][ldS] (bands * 18 columns), frames: [rows][bands*16].  4 rows per CTA, 64 threads per row.
__global__ void __launch_bounds__(256) istft_frames_kernel(const float* __restrict__ s, int ldS,
                                                            float* __restrict__ frames, int rows, int bands) {
    // 7 rows per CTA: phase 1 uses 7*36 = 252 threads (one per (row, band, bin)) for the transcendental
    // work, phase 2 uses 64 threads per row for the 16-point inverse real DFT + window.
    constexpr int RPB = 7;
    __shared__ float re[RPB][4][9], im[RPB][4][9];
    // twiddle / window tables in SHARED memory: the index varies per lane, and divergent __constant__
    // reads serialise (this kernel took 1.65 ms per step with constant-memory tables)
    __shared__ float s_cos[16], s_sin[16], s_hann[16];
    if (threadIdx.x < 16) { s_cos[threadIdx.x] = c_cos16[threadIdx.x]; s_sin[threadIdx.x] = c_sin16[threadIdx.x]; s_hann[threadIdx.x] = c_hann[threadIdx.x]; }
    const int row0 = blockIdx.x * RPB;
    {
        const int rl = threadIdx.x / 36, q = threadIdx.x - rl * 36;
        const int row = row0 + rl;
        if (rl < RPB && row < rows && q < bands * 9) {
            const int b = q / 9, k = q - b * 9;
            const float mag = expf(s[(size_t)row * ldS + b * 18 + k]);
            const float ph = sinf(s[(size_t)row * ldS + b * 18 + 9 + k]) * 3.14159265358979323846f;
            float sn, cs;
            sincosf(ph, &sn, &cs);
            re[rl][b][k] = mag * cs;
            im[rl][b][k] = mag * sn;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < RPB * 64; e += 256) {
        const int rl = e >> 6, q = e & 63;
        const int row = row0 + rl;
        if (row >= rows || q >= bands * 16) continue;
        const int b = q >> 4, n = q & 15;
        float acc = 0.f;
#pragma unroll
        for (int k = 1; k < 8; ++k) {
            const int mI = (k * n) & 15;
            acc += re[rl][b][k] * s_cos[mI] - im[rl][b][k] * s_sin[mI];
        }
        const float x = (re[rl][b][0] + ((n & 1) ? -re[rl][b][8] : re[rl][b][8]) + 2.0f * acc) * (1.0f / 16.0f);
        frames[(size_t)row * (bands * 16) + q] = x * s_hann[n];
    }
}

// K12. overlap-add (hop 4) + window-sum normalisation + centre crop: iStft.cpp:99-123.
// yb[i][b], i in [0, 4*(rows_u-1)) per utterance.  sfr: frame rows (len_u = 16F+1), sy: rate 4x.
__global__ void istft_ola_kernel(const float* __restrict__ frames, float* __restrict__ yb, Seg sfr, Seg sy, int bands) {
    __shared__ float s_hp[16];
    if (threadIdx.x < 16) s_hp[threadIdx.x] = c_hann_pow[threadIdx.x];
    __syncthreads();
    const int u = blockIdx.y;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int nfr = seg_len(sfr, u);
    const int ny = seg_len(sy, u);
    if (idx >= ny * bands) return;
    const int i = idx / bands, b = idx % bands;
    const int pos = i + 8;
    float acc = 0.f, ws = 0.f;
    int jlo = (pos - 15 + 3) >> 2;
    if (jlo < 0) jlo = 0;
    int jhi = pos >> 2;
    if (jhi > nfr - 1) jhi = nfr - 1;
    const int f0 = seg_start(sfr, u);
    for (int j = jlo; j <= jhi; ++j) {
        const int n = pos - 4 * j;
        acc += frames[(size_t)(f0 + j) * (bands * 16) + b * 16 + n];
        ws += s_hp[n];
    }
    if (ws > 1e-14f) acc = acc / ws;
    yb[(size_t)(seg_start(sy, u) + i) * bands + b] = acc;
}

// K13. zero-stuff x4 (gain 4) + 63-tap synthesis FIR (learned multistream_conv_post or PQMF):
// Generator_MS.cpp:106-124,225-226 / pqmf.cpp:97-115.  Only every 4th tap hits a non-zero sample.
// yb: [n][4]; w: [63][4] (tap-major); out o[s], s in [0, 4n).
__global__ void __launch_bounds__(256) synth_fir_kernel(const float* __restrict__ yb, const float* __restrict__ w,
                                                         const float* __restrict__ bias, float* __restrict__ o,
                                                         Seg sy, Seg so) {
    __shared__ float ws[63 * 4];
    for (int i = threadIdx.x; i < 63 * 4; i += blockDim.x) ws[i] = w[i];
    __syncthreads();
    const int u = blockIdx.y;
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int ns = seg_len(so, u);
    if (s >= ns) return;
    const int ny = seg_len(sy, u);
    const int y0 = seg_start(sy, u);
    float acc = 0.f;
    const int k0 = ((31 - s) % 4 + 4) % 4;
    for (int k = k0; k < 63; k += 4) {
        const int p = s + k - 31;
        if (p < 0) continue;
        const int i = p >> 2;
        if (i >= ny) break;
        const float4 v = *reinterpret_cast<const float4*>(yb + (size_t)(y0 + i) * 4);
        acc = fmaf(v.x * 4.0f, ws[k * 4 + 0], acc);
        acc = fmaf(v.y * 4.0f, ws[k * 4 + 1], acc);
        acc = fmaf(v.z * 4.0f, ws[k * 4 + 2], acc);
        acc = fmaf(v.w * 4.0f, ws[k * 4 + 3], acc);
    }
    if (bias) acc += bias[0];
    o[(size_t)seg_start(so, u) + s] = acc;
}

// K14. float waveform -> int16 PCM: retData[i] = (int16_t)(o[i]*32737), SynthesizerTrn.cpp:389-396
// (truncation toward zero, no clipping; the constant is 32737 in the reference).
__global__ void pcm_kernel(const float* __restrict__ o, int16_t* __restrict__ pcm, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) pcm[i] = (int16_t)__float2int_rz(o[i] * 32737.0f);
}

// K15. The whole 4-band tail in one launch: K11 + K12 + K13 + K14 over a tile of TI band samples with the halos each stage needs,
// all intermediates in shared memory (round 1 wrote and re-read frames [rows][64], yb [4 rows][4] and o through HBM in four
// launches).  Same arithmetic, same order: bit-identical to the four kernels.  Generator_MS.cpp:210-229 / Generator_MBB.cpp:176-203,
// iStft.cpp:63-123, SynthesizerTrn.cpp:389-396.
template <int MT_TI>                             // band samples per CTA (-> 4 MT_TI output samples)
__global__ void __launch_bounds__(256) ms_tail_kernel(const float* __restrict__ sp, int ldS, const float* __restrict__ w, const float* __restrict__ bias,
                                                       float* __restrict__ o, int16_t* __restrict__ pcm, Seg sfr, Seg sy, Seg so) {
    constexpr int MT_NF = MT_TI / 4 + 8;          // frame rows a tile touches
    extern __shared__ __align__(16) float mtsm[];
    float* re = mtsm;                             // [MT_NF][36]
    float* im = re + MT_NF * 36;                  // [MT_NF][36]
    float* fr = im + MT_NF * 36;                  // [MT_NF][64]
    float* ybs = fr + MT_NF * 64;                 // [MT_TI + 16][4]
    float* wsm = ybs + (MT_TI + 16) * 4;          // [63][4]
    __shared__ float s_cos[16], s_sin[16], s_hann[16], s_hp[16];
    const int u = blockIdx.y;
    const int ny = seg_len(sy, u);
    const int i0 = blockIdx.x * MT_TI;
    if (i0 >= ny) return;
    const int nfr = seg_len(sfr, u), f0 = seg_start(sfr, u);
    const int tid = threadIdx.x;
    if (tid < 16) { s_cos[tid] = c_cos16[tid]; s_sin[tid] = c_sin16[tid]; s_hann[tid] = c_hann[tid]; s_hp[tid] = c_hann_pow[tid]; }
    for (int i = tid; i < 63 * 4; i += 256) wsm[i] = w[i];
    const int jbase = (i0 - 12) >> 2;             // first frame row of the tile (arithmetic shift: may be negative)
    // ---- K11 phase 1: exp / pi*sin -> complex bins ---------------------------------------------------
    for (int e = tid; e < MT_NF * 36; e += 256) {
        const int jl = e / 36, q = e - jl * 36;
        const int j = jbase + jl;
        float r_ = 0.f, i_ = 0.f;
        if (j >= 0 && j < nfr) {
            const int b = q / 9, k = q - b * 9;
            const float* row = sp + (size_t)(f0 + j) * ldS + b * 18;
            const float mag = expf(row[k]);
            const float ph = sinf(row[9 + k]) * 3.14159265358979323846f;
            float sn, cs;
            sincosf(ph, &sn, &cs);
            r_ = mag * cs; i_ = mag * sn;
        }
        re[e] = r_; im[e] = i_;
    }
    __syncthreads();
    // ---- K11 phase 2: 16-point real inverse DFT + window --------------------------------------------
    for (int e = tid; e < MT_NF * 64; e += 256) {
        const int jl = e >> 6, q = e & 63;
        const int b = q >> 4, n = q & 15;
        const float* rr = re + jl * 36 + b * 9;
        const float* ii = im + jl * 36 + b * 9;
        float acc = 0.f;
#pragma unroll
        for (int k = 1; k < 8; ++k) {
            const int mI = (k * n) & 15;
            acc += rr[k] * s_cos[mI] - ii[k] * s_sin[mI];
        }
        const float x = (rr[0] + ((n & 1) ? -rr[8] : rr[8]) + 2.0f * acc) * (1.0f / 16.0f);
        fr[e] = x * s_hann[n];
    }
    __syncthreads();
    // ---- K12: overlap-add + window-sum normalisation + centre crop ------------------------------------
    for (int e = tid; e < (MT_TI + 16) * 4; e += 256) {
        const int il = e >> 2, b = e & 3;
        const int i = i0 - 8 + il;
        float acc = 0.f;
        if (i >= 0 && i < ny) {
            const int pos = i + 8;
            float wsum = 0.f;
            int jlo = (pos - 15 + 3) >> 2;
            if (jlo < 0) jlo = 0;
            int jhi = pos >> 2;
            if (jhi > nfr - 1) jhi = nfr - 1;
            for (int j = jlo; j <= jhi; ++j) {
                const int n = pos - 4 * j;
                acc += fr[(j - jbase) * 64 + b * 16 + n];
                wsum += s_hp[n];
            }
            if (wsum > 1e-14f) acc = acc / wsum;
        }
        ybs[e] = acc;
    }
    __syncthreads();
    // ---- K13 + K14: zero-stuff x4 (gain 4) + 63-tap synthesis FIR, float waveform + int16 PCM ----------
    const int ns = seg_len(so, u);
    const size_t s0 = (size_t)seg_start(so, u);
    for (int sl = tid; sl < 4 * MT_TI; sl += 256) {
        const int sidx = 4 * i0 + sl;
        if (sidx >= ns) break;
        float acc = 0.f;
        const int k0 = ((31 - sidx) % 4 + 4) % 4;
        for (int k = k0; k < 63; k += 4) {
            const int p = sidx + k - 31;
            if (p < 0) continue;
            const int i = p >> 2;
            if (i >= ny) break;
            const float4 v = *reinterpret_cast<const float4*>(ybs + (size_t)(i - (i0 - 8)) * 4);
            acc = fmaf(v.x * 4.0f, wsm[k * 4 + 0], acc);
            acc = fmaf(v.y * 4.0f, wsm[k * 4 + 1], acc);
            acc = fmaf(v.z * 4.0f, wsm[k * 4 + 2], acc);
            acc = fmaf(v.w * 4.0f, wsm[k * 4 + 3], acc);
        }
        if (bias) acc += bias[0];
        o[s0 + sidx] = acc;
        pcm[s0 + sidx] = (int16_t)__float2int_rz(acc * 32737.0f);
    }
}
inline size_t ms_tail_smem(int ti) { const size_t nf = ti / 4 + 8; return (nf * 36 * 2 + nf * 64 + (size_t)(ti + 16) * 4 + 63 * 4) * sizeof(float); }

// column 0 copy (Generator_Istft: single band -> waveform)
__global__ void copy_kernel(const float* __restrict__ a, float* __restrict__ b, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) b[i] = a[i];
}

}  // namespace stts
