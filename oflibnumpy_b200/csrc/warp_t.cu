// Target-referenced (backward) warp for sm_100a: bilinear gather with OpenCV's 1/32-px fixed-point coordinates,
// payload and validity mask resampled in the same pass. Replaces cv2.remap at utils.py:236 of the reference plus the
// mask plumbing of Flow.apply (flow_class.py:631-680). HBM-bound gather: no tensor cores.
//
// Two kernels:
//   warp_t_rows    a warp owns 32 consecutive pixels of a row and walks 4 rows (CTA = 32x32 tile): every access of a
//                  warp instruction is contiguous along x, the gathered neighbourhood of a tile stays in L1.
//   warp_t_u8x3    the image case: both horizontal taps of a row come from one aligned 64-bit load, the horizontal
//                  blend runs on packed bytes (dp4a), rounding is integer, 96-byte rows are stored as 24 words.
//   warp_t_generic 1 pixel per thread, any channel count / dtype / padding offsets / unaligned pointers.
#include <algorithm>

#include "ofk_common.cuh"
#include "warp_t_device.cuh"

namespace ofk {

enum : int { AR_U8_FIXED = 0, AR_RINT = 1, AR_F32 = 2, AR_F64 = 3 };

template <typename T>
__device__ __forceinline__ T saturate_rint(float v);
template <>
__device__ __forceinline__ uint8_t saturate_rint<uint8_t>(float v) {
    return static_cast<uint8_t>(max(0, min(255, __float2int_rn(v))));
}
template <>
__device__ __forceinline__ int16_t saturate_rint<int16_t>(float v) {
    return static_cast<int16_t>(max(-32768, min(32767, __float2int_rn(v))));
}
template <>
__device__ __forceinline__ uint16_t saturate_rint<uint16_t>(float v) {
    return static_cast<uint16_t>(max(0, min(65535, __float2int_rn(v))));
}
template <>
__device__ __forceinline__ float saturate_rint<float>(float v) {
    return v;
}
template <>
__device__ __forceinline__ double saturate_rint<double>(float v) {
    return v;
}

// One interpolated value from four taps, in OpenCV's arithmetic for the given mode (sums left to right, no FMA
// contraction: cv2.remap's results are reproduced bit for bit, see tests/test_oracle_remap.py for the CPU statement).
template <typename T, int AR>
__device__ __forceinline__ T blend(T t00, T t01, T t10, T t11, const QWeights& w) {
    if (AR == AR_U8_FIXED) {
        // (sum t*w*32 + 2^14) >> 15 with 15-bit weights w*32  ==  (sum t*w + 512) >> 10
        int acc = int(t00) * w.w00 + int(t01) * w.w01 + int(t10) * w.w10 + int(t11) * w.w11;
        return static_cast<T>((acc + 512) >> 10);
    } else if (AR == AR_F64) {
        const double s = 1.0 / 1024.0;
        double acc = __dmul_rn(double(t00), double(w.w00) * s);
        acc = __dadd_rn(acc, __dmul_rn(double(t01), double(w.w01) * s));
        acc = __dadd_rn(acc, __dmul_rn(double(t10), double(w.w10) * s));
        acc = __dadd_rn(acc, __dmul_rn(double(t11), double(w.w11) * s));
        return static_cast<T>(acc);
    } else {
        const float s = 1.0f / 1024.0f;  // weights are exact multiples of 2^-10
        float acc = __fmul_rn(float(t00), float(w.w00) * s);
        acc = __fadd_rn(acc, __fmul_rn(float(t01), float(w.w01) * s));
        acc = __fadd_rn(acc, __fmul_rn(float(t10), float(w.w10) * s));
        acc = __fadd_rn(acc, __fmul_rn(float(t11), float(w.w11) * s));
        if (AR == AR_RINT) return saturate_rint<T>(acc);
        return static_cast<T>(acc);
    }
}

struct Taps {
    int ix, iy;
    QWeights w;
    bool in00, in01, in10, in11;
    bool interior;
};

__device__ __forceinline__ Taps make_taps(float X, float Y, int Hs, int Ws) {
    QCoord qx = quantise(X), qy = quantise(Y);
    Taps t;
    t.ix = qx.i;
    t.iy = qy.i;
    t.w = qweights(qx.f, qy.f);
    bool x0 = (unsigned)t.ix < (unsigned)Ws, x1 = (unsigned)(t.ix + 1) < (unsigned)Ws;
    bool y0 = (unsigned)t.iy < (unsigned)Hs, y1 = (unsigned)(t.iy + 1) < (unsigned)Hs;
    t.in00 = x0 && y0;
    t.in01 = x1 && y0;
    t.in10 = x0 && y1;
    t.in11 = x1 && y1;
    t.interior = t.in00 && t.in11;
    return t;
}

// valid-weight sum in 1/1024 units; pm == nullptr means "payload everywhere valid" (only bounds matter)
__device__ __forceinline__ int valid_weight_sum(const Taps& t, const uint8_t* __restrict__ pm, int Ws) {
    int S = 0;
    if (pm == nullptr) {
        S = (t.in00 ? t.w.w00 : 0) + (t.in01 ? t.w.w01 : 0) + (t.in10 ? t.w.w10 : 0) + (t.in11 ? t.w.w11 : 0);
    } else {
        const long long o = (long long)t.iy * Ws + t.ix;
        if (t.in00 && pm[o]) S += t.w.w00;
        if (t.in01 && pm[o + 1]) S += t.w.w01;
        if (t.in10 && pm[o + Ws]) S += t.w.w10;
        if (t.in11 && pm[o + Ws + 1]) S += t.w.w11;
    }
    return S;
}

// ----------------------------------------------------------------------------------------------- generic kernel
template <typename T, int AR>
__global__ void __launch_bounds__(256) warp_t_generic(const T* __restrict__ payload, int C,
                                                      const float* __restrict__ flow, float sign,
                                                      const uint8_t* __restrict__ pmask,
                                                      const uint8_t* __restrict__ fmask, T* __restrict__ out,
                                                      uint8_t* __restrict__ omask, int rule, int H, int W, int Hs,
                                                      int Ws, int Ho, int Wo, int oy, int ox, int fy, int fx) {
    // output frame (Ho, Wo); output pixel (y, x) sits at (y + oy, x + ox) of the payload frame and at
    // (y - fy, x - fx) of the flow frame (zero flow / invalid outside it).
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int n = blockIdx.z;
    if (x >= Wo || y >= Ho) return;
    const int yf = y - fy, xf = x - fx;
    const bool in_flow = (unsigned)yf < (unsigned)H && (unsigned)xf < (unsigned)W;
    float u = 0.f, v = 0.f;
    if (in_flow) {
        const float* f = flow + (((size_t)n * H + yf) * W + xf) * 2;
        u = f[0];
        v = f[1];
    }
    const float X = sample_coord(u, sign, x + ox);
    const float Y = sample_coord(v, sign, y + oy);
    const Taps t = make_taps(X, Y, Hs, Ws);
    const size_t opix = ((size_t)n * Ho + y) * Wo + x;
    if (omask != nullptr) {
        const uint8_t* pm = pmask ? pmask + (size_t)n * Hs * Ws : nullptr;
        bool ok = mask_rule_pass(valid_weight_sum(t, pm, Ws), rule);
        if (!in_flow) ok = false;
        else if (fmask) ok = ok && fmask[((size_t)n * H + yf) * W + xf];
        omask[opix] = ok ? 1 : 0;
    }
    if (C > 0) {
        const T* p = payload + (size_t)n * Hs * Ws * C;
        const long long o = ((long long)t.iy * Ws + t.ix) * C;
        const long long row = (long long)Ws * C;
        for (int c = 0; c < C; ++c) {
            T t00 = t.in00 ? p[o + c] : T(0);
            T t01 = t.in01 ? p[o + C + c] : T(0);
            T t10 = t.in10 ? p[o + row + c] : T(0);
            T t11 = t.in11 ? p[o + row + C + c] : T(0);
            out[opix * C + c] = blend<T, AR>(t00, t01, t10, t11, t.w);
        }
    }
}

// ----------------------------------------------------------------------------------------------- rows kernel
// Thread mapping: a warp owns 32 consecutive pixels of a row (lane = x) and walks 4 rows, a CTA owns a 32x32 tile.
// Every global access of a warp instruction is therefore contiguous along x: flow / mask / output are fully
// coalesced and the gathers of a warp touch 2-3 cache lines (a rotated row segment) instead of 8.

// Per-(T,C) tap fetch for one pixel: fills v[4][C] (tap order 00,01,10,11) with zero for out-of-bounds taps.
template <typename T, int C>
struct Fetch {
    __device__ __forceinline__ static void run(const T* __restrict__ p, int Ws, const Taps& t, T (&v)[4][C]) {
        const int o = (t.iy * Ws + t.ix) * C, row = Ws * C;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            v[0][c] = t.in00 ? __ldg(p + o + c) : T(0);
            v[1][c] = t.in01 ? __ldg(p + o + C + c) : T(0);
            v[2][c] = t.in10 ? __ldg(p + o + row + c) : T(0);
            v[3][c] = t.in11 ? __ldg(p + o + row + C + c) : T(0);
        }
    }
};

// float32 x2 (flow fields): one 64-bit load per tap
template <>
struct Fetch<float, 2> {
    __device__ __forceinline__ static void run(const float* __restrict__ p, int Ws, const Taps& t, float (&v)[4][2]) {
        const float2* q = reinterpret_cast<const float2*>(p);
        const int o = t.iy * Ws + t.ix;
        const float2 z = make_float2(0.f, 0.f);
        const float2 a = t.in00 ? __ldg(q + o) : z;
        const float2 b = t.in01 ? __ldg(q + o + 1) : z;
        const float2 c = t.in10 ? __ldg(q + o + Ws) : z;
        const float2 d = t.in11 ? __ldg(q + o + Ws + 1) : z;
        v[0][0] = a.x; v[0][1] = a.y;
        v[1][0] = b.x; v[1][1] = b.y;
        v[2][0] = c.x; v[2][1] = c.y;
        v[3][0] = d.x; v[3][1] = d.y;
    }
};

// float32 x4: one 128-bit load per tap
template <>
struct Fetch<float, 4> {
    __device__ __forceinline__ static void run(const float* __restrict__ p, int Ws, const Taps& t, float (&v)[4][4]) {
        const float4* q = reinterpret_cast<const float4*>(p);
        const int o = t.iy * Ws + t.ix;
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 r[4] = {t.in00 ? __ldg(q + o) : z, t.in01 ? __ldg(q + o + 1) : z, t.in10 ? __ldg(q + o + Ws) : z,
                             t.in11 ? __ldg(q + o + Ws + 1) : z};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[k][0] = r[k].x; v[k][1] = r[k].y; v[k][2] = r[k].z; v[k][3] = r[k].w;
        }
    }
};

// uint8 x4: one 32-bit load per tap
template <>
struct Fetch<uint8_t, 4> {
    __device__ __forceinline__ static void run(const uint8_t* __restrict__ p, int Ws, const Taps& t,
                                               uint8_t (&v)[4][4]) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
        const int o = t.iy * Ws + t.ix;
        uint32_t w[4];
        w[0] = t.in00 ? __ldg(q + o) : 0u;
        w[1] = t.in01 ? __ldg(q + o + 1) : 0u;
        w[2] = t.in10 ? __ldg(q + o + Ws) : 0u;
        w[3] = t.in11 ? __ldg(q + o + Ws + 1) : 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            v[k][0] = w[k] & 0xff;
            v[k][1] = (w[k] >> 8) & 0xff;
            v[k][2] = (w[k] >> 16) & 0xff;
            v[k][3] = w[k] >> 24;
        }
    }
};

// Store C elements of one pixel (contiguous across the warp).
template <typename T, int C>
__device__ __forceinline__ void store_px(T* __restrict__ dst, const T (&r)[C]) {
    if constexpr (sizeof(T) * C == 8) {
        uint2 u;
        memcpy(&u, r, 8);
        *reinterpret_cast<uint2*>(dst) = u;
    } else if constexpr (sizeof(T) * C == 16) {
        uint4 u;
        memcpy(&u, r, 16);
        *reinterpret_cast<uint4*>(dst) = u;
    } else if constexpr (sizeof(T) * C == 4) {
        uint32_t u;
        memcpy(&u, r, 4);
        *reinterpret_cast<uint32_t*>(dst) = u;
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) dst[c] = r[c];
    }
}

template <typename T, int C, int AR>
__global__ void __launch_bounds__(256) warp_t_rows(const T* __restrict__ payload, const float* __restrict__ flow,
                                                   float sign, const uint8_t* __restrict__ pmask,
                                                   const uint8_t* __restrict__ fmask, T* __restrict__ out,
                                                   uint8_t* __restrict__ omask, int rule, int H, int W) {
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const int x = blockIdx.x * 32 + lane;
    const int y0 = blockIdx.y * 32 + wrp * 4;
    const size_t frame = (size_t)H * W, fbase = (size_t)blockIdx.z * frame;
    if (x >= W) return;
    const float2* fl = reinterpret_cast<const float2*>(flow) + fbase;
    const uint8_t* fm = fmask ? fmask + fbase : nullptr;
    const uint8_t* pm = pmask ? pmask + fbase : nullptr;
    const T* p = C > 0 ? payload + fbase * C : nullptr;
    const float Xg = static_cast<float>(x);
    float2 f[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (y0 + j < H) f[j] = ld_stream_f2(fl + (y0 + j) * W + x);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int y = y0 + j;
        if (y >= H) break;
        const int pix = y * W + x;
        const Taps t = make_taps(__fadd_rn(sign * f[j].x, Xg), __fadd_rn(sign * f[j].y, static_cast<float>(y)), H, W);
        if constexpr (C > 0) {
            T taps[4][C], res[C];
            Fetch<T, C>::run(p, W, t, taps);
#pragma unroll
            for (int c = 0; c < C; ++c) res[c] = blend<T, AR>(taps[0][c], taps[1][c], taps[2][c], taps[3][c], t.w);
            store_px<T, C>(out + (fbase + pix) * C, res);
        }
        if (omask != nullptr) {
            const int S = (pm == nullptr && t.interior) ? 1024 : valid_weight_sum(t, pm, W);
            const bool ok = mask_rule_pass(S, rule) && (fm == nullptr || fm[pix] != 0);
            omask[fbase + pix] = ok ? 1 : 0;
        }
    }
}

// ------------------------------------------------------------------------------------- uint8 x3 (images), specialised
// Both arithmetic modes are pure integer for 8-bit taps: with weights k/1024 the float32 products and partial sums of
// cv2.remap's int16 path are exact (< 2^18 in units of 1/1024), so cvRound(sum) == round-half-even(acc / 1024) where
// acc = sum t*w is the same integer the fixed-point path rounds half-up.
__device__ __forceinline__ uint32_t round_acc(int acc, bool half_even) {
    return half_even ? (uint32_t)(acc + 511 + ((acc >> 10) & 1)) >> 10 : (uint32_t)(acc + 512) >> 10;
}

// bytes [b0..b5] at byte offset `off` from the 4-byte aligned base pa (the two horizontal taps of a row):
// lo = b0..b3, hi = b4,b5 (upper half undefined). Three aligned 32-bit loads off one address, two funnel shifts.
__device__ __forceinline__ void window6(const uint8_t* __restrict__ pa, int off, uint32_t& lo, uint32_t& hi) {
    const uint32_t* q = reinterpret_cast<const uint32_t*>(pa + (off & ~3));
    const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
    const unsigned t = (unsigned)off << 3;          // funnel shift uses t & 31 = 8 * (off & 3)
    lo = __funnelshift_r(w0, w1, t);
    hi = __funnelshift_r(w1, w2, t);
}

// bytes [b0..b5] at byte offset `off` from the 4-byte aligned base pa (the two horizontal taps of a row):
// lo = b0..b3, hi = b4,b5 (upper half undefined). Three aligned 32-bit loads off one address, two funnel shifts.
__device__ __forceinline__ void window6(const uint8_t* __restrict__ pa, unsigned off, uint32_t& lo, uint32_t& hi) {
    const uint32_t* q = reinterpret_cast<const uint32_t*>(pa + (off & ~3u));
    const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
    const unsigned t = off << 3;                    // funnel shift uses t & 31 = 8 * (off & 3)
    lo = __funnelshift_r(w0, w1, t);
    hi = __funnelshift_r(w1, w2, t);
}

// HALF_EVEN: cv2.remap's int16 path (cvRound) instead of the uint8 fixed-point path; PM: a payload mask is resampled.
// Loads use clamped indices (no branches), only the stores are predicated.
template <bool HALF_EVEN, bool PM>
__global__ void __launch_bounds__(256) warp_t_u8x3(const uint8_t* __restrict__ payload,
                                                   const float* __restrict__ flow, float sign,
                                                   const uint8_t* __restrict__ pmask,
                                                   const uint8_t* __restrict__ fmask, uint8_t* __restrict__ out,
                                                   uint8_t* __restrict__ omask, int rule, int H, int W,
                                                   int packed_store) {
    const unsigned lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const unsigned x = blockIdx.x * 32 + lane, xc = min(x, (unsigned)W - 1);
    const unsigned y0 = blockIdx.y * 32 + wrp * 4;
    const size_t frame = (size_t)H * W, fbase = (size_t)blockIdx.z * frame;
    const bool full_row = packed_store && (blockIdx.x * 32 + 32 <= (unsigned)W);   // warp-uniform
    const float2* fl = reinterpret_cast<const float2*>(flow) + fbase;
    const uint8_t* fm = fmask ? fmask + fbase : nullptr;
    const uint8_t* pm = PM ? pmask + fbase : nullptr;
    const uint8_t* p = payload + fbase * 3;
    // 4-byte aligned view of the frame for the word loads of the interior path
    const unsigned r0 = (unsigned)(reinterpret_cast<uintptr_t>(p) & 3);
    const uint8_t* pa = p - r0;
    const size_t avail = (size_t)(payload + (size_t)gridDim.z * frame * 3 - pa);
    const unsigned limit = avail > 0x7fffffffu ? 0x7fffffffu : (unsigned)avail;
    uint8_t* o = out + fbase * 3;
    uint8_t* om = omask ? omask + fbase : nullptr;
    const float Xg = static_cast<float>(x);
    const unsigned row3 = (unsigned)W * 3;
    float2 f[4];
    unsigned fmv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned idx = min(y0 + j, (unsigned)H - 1) * (unsigned)W + xc;
        f[j] = ld_stream_f2(fl + idx);
        fmv[j] = (om != nullptr && fm != nullptr) ? fm[idx] : 1u;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned y = y0 + j;
        if (y >= (unsigned)H) break;                                     // warp-uniform
        const float X = __fmaf_rn(sign, f[j].x, Xg), Y = __fmaf_rn(sign, f[j].y, static_cast<float>(y));
        const QCoord qx = quantise_fast(X), qy = quantise_fast(Y);
        const unsigned off = (unsigned)(qy.i * W + qx.i) * 3 + r0;
        const bool interior = (unsigned)qx.i < (unsigned)(W - 1) && (unsigned)qy.i < (unsigned)(H - 1) &&
                              fabsf(X) < OFK_FAST_COORD_LIMIT && fabsf(Y) < OFK_FAST_COORD_LIMIT &&
                              off + row3 + 12 <= limit;
        uint32_t v;
        unsigned ok;
        if (interior) {
            uint32_t lo0, hi0, lo1, hi1;
            window6(pa, off, lo0, hi0);
            window6(pa, off + row3, lo1, hi1);
            const uint32_t a = qx.f, na = 32 - a;
            const int b = qy.f;
            ok = 1;
            if (PM) {
                const uint8_t* m0 = pm + (unsigned)(qy.i * W + qx.i);
                const uint8_t* m1 = m0 + W;
                const QWeights w = qweights((int)a, b);
                const int S = (m0[0] ? w.w00 : 0) + (m0[1] ? w.w01 : 0) + (m1[0] ? w.w10 : 0) + (m1[1] ? w.w11 : 0);
                ok = mask_rule_pass(S, rule);
            }
            // horizontal pass with 8-bit weights on packed bytes (dp4a); vertical pass in 32 bits with the weights
            // scaled by 64 so the rounded result lands in byte 2: t = acc * 64 + 512 * 64
            const uint32_t w0 = na | (a << 24);                     // ch0: lo byte0 (tap 0) and lo byte3 (tap 1)
            const uint32_t w1l = na << 8, w1h = a;                  // ch1: lo byte1, hi byte0
            const uint32_t w2l = na << 16, w2h = a << 8;            // ch2: lo byte2, hi byte1
            const uint32_t vb = (uint32_t)b << 6, vnb = 2048u - vb;
            const uint32_t t0 = __dp4a(lo0, w0, 0u) * vnb + (__dp4a(lo1, w0, 0u) * vb + 32768u);
            const uint32_t t1 = __dp4a(lo0, w1l, __dp4a(hi0, w1h, 0u)) * vnb +
                                (__dp4a(lo1, w1l, __dp4a(hi1, w1h, 0u)) * vb + 32768u);
            const uint32_t t2 = __dp4a(lo0, w2l, __dp4a(hi0, w2h, 0u)) * vnb +
                                (__dp4a(lo1, w2l, __dp4a(hi1, w2h, 0u)) * vb + 32768u);
            // round half up = byte 2 of t; bytes: v = [t0.b2, t1.b2, t2.b2, 0]
            v = __byte_perm(__byte_perm(t0, t1, 0x0062), t2, 0x4610) & 0x00ffffffu;
            if (HALF_EVEN) {
                // cvRound sends exact ties to the even neighbour: a tie that rounded up to an odd value shows as
                // (t & 0x1ffff) == 0x10000. Rare, so test all three at once and fix up out of the main flow.
                const uint32_t m0 = (t0 & 0x1ffffu) ^ 0x10000u, m1 = (t1 & 0x1ffffu) ^ 0x10000u,
                               m2 = (t2 & 0x1ffffu) ^ 0x10000u;
                if (min(m0, min(m1, m2)) == 0u) {
                    if (m0 == 0u) v -= 1u;
                    if (m1 == 0u) v -= 1u << 8;
                    if (m2 == 0u) v -= 1u << 16;
                }
            }
        } else {
            const uint32_t r = border_px_u8x3(p, pm, X, Y, H, W, HALF_EVEN, rule);
            v = r & 0x00ffffffu;
            ok = r >> 24;
        }
        const bool xin = x < (unsigned)W;
        if (om != nullptr && xin) om[y * (unsigned)W + x] = (uint8_t)(ok & fmv[j]);
        if (full_row) {
            // 32 pixels x 3 bytes = 24 words: lane L < 24 assembles word L from pixels L + L/3 and the next one
            const unsigned p0 = lane + lane / 3;
            const uint32_t v0 = __shfl_sync(0xffffffffu, v, p0 & 31), v1 = __shfl_sync(0xffffffffu, v, (p0 + 1) & 31);
            const uint32_t word = __funnelshift_r(v0 | (v1 << 24), v1 >> 8, 8 * (lane % 3));
            if (lane < 24)
                st_stream_u32(reinterpret_cast<uint32_t*>(o + ((size_t)y * W + blockIdx.x * 32) * 3) + lane, word);
        } else if (xin) {
            uint8_t* d = o + ((size_t)y * W + x) * 3;
            d[0] = (uint8_t)v;
            d[1] = (uint8_t)(v >> 8);
            d[2] = (uint8_t)(v >> 16);
        }
    }
}


// ------------------------------------------------------------------------------------- valid area without payload
// valid_target (ref 't') / valid_source (ref 's'), flow_class.py:1148-1150,1179-1183: "every tap with a non-zero
// weight lies inside the frame", AND the flow mask. Pure streaming (8 + 1 B/px in, 1 B/px out): 4 consecutive pixels
// per thread, 2 x 16-byte flow loads, one 32-bit mask word in and out.
__global__ void __launch_bounds__(256) valid_geom_vec4(const float4* __restrict__ flow, float sign,
                                                       const uint32_t* __restrict__ fmask, uint32_t* __restrict__ out,
                                                       int H, int W, unsigned quads_per_frame) {
    const unsigned r = blockIdx.x * blockDim.x + threadIdx.x;      // quad index inside frame blockIdx.y
    if (r >= quads_per_frame) return;
    const size_t q = (size_t)blockIdx.y * quads_per_frame + r;
    const unsigned wq = (unsigned)W >> 2;
    const int y = (int)(r / wq), x = (int)(r - (unsigned)y * wq) << 2;
    const float4 f0 = ld_stream_f4(flow + 2 * q), f1 = ld_stream_f4(flow + 2 * q + 1);
    const uint32_t m = fmask ? ld_stream_u32(fmask + q) : 0x01010101u;
    const float Yg = (float)y;
    uint32_t v = strict_in_frame(__fmaf_rn(sign, f0.x, (float)x), __fmaf_rn(sign, f0.y, Yg), H, W);
    v |= strict_in_frame(__fmaf_rn(sign, f0.z, (float)(x + 1)), __fmaf_rn(sign, f0.w, Yg), H, W) << 8;
    v |= strict_in_frame(__fmaf_rn(sign, f1.x, (float)(x + 2)), __fmaf_rn(sign, f1.y, Yg), H, W) << 16;
    v |= strict_in_frame(__fmaf_rn(sign, f1.z, (float)(x + 3)), __fmaf_rn(sign, f1.w, Yg), H, W) << 24;
    st_stream_u32(out + q, v & m);
}

// apply_flow returns its target untouched for a flow that is zero below the threshold (utils.py:215-216). The warp's
// identity taps reproduce that for integer payloads but not for floats: NaN / Inf on a zero-weight tap poison the
// result, and -0.0 next to a positive value comes out as +0. Frames whose flag is 0 get the payload copied over the
// warp's output (bit for bit: E is an unsigned type of the element size). The valid area needs no repair: with identity
// taps it already is the mask that went in, ANDed with the flow mask.
template <typename E>
__global__ void __launch_bounds__(256) warp_t_passthrough(const E* __restrict__ payload, const int* __restrict__ nz,
                                                          E* __restrict__ out, int Ho, long long rowlen,
                                                          long long src_row, long long src_off, long long src_frame) {
    const int n = blockIdx.z;
    if (nz[n]) return;
    const E* src = payload + n * src_frame + src_off;
    E* dst = out + (long long)n * Ho * rowlen;
    for (long long y = blockIdx.y; y < Ho; y += gridDim.y)
        for (long long i = blockIdx.x * 256ll + threadIdx.x; i < rowlen; i += gridDim.x * 256ll)
            dst[y * rowlen + i] = src[y * src_row + i];
}

template <typename T, int C, int AR>
static int launch_rows(const void* payload, const float* flow, float sign, const uint8_t* pmask, const uint8_t* fmask,
                       void* out, uint8_t* omask, int rule, int N, int H, int W, cudaStream_t st) {
    dim3 grid((W + 31) / 32, (H + 31) / 32, N);
    warp_t_rows<T, C, AR><<<grid, 256, 0, st>>>(static_cast<const T*>(payload), flow, sign, pmask, fmask,
                                                static_cast<T*>(out), omask, rule, H, W);
    OFK_LAUNCHED();
    return OFK_OK;
}

static int launch_u8x3(bool half_even, const void* payload, const float* flow, float sign, const uint8_t* pmask,
                       const uint8_t* fmask, void* out, uint8_t* omask, int rule, int N, int H, int W,
                       cudaStream_t st) {
    dim3 grid((W + 31) / 32, (H + 31) / 32, N);
    // word stores need every row start 4-byte aligned: W % 4 == 0 and a 4-byte aligned base
    const int packed = (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 3) == 0);
#define OFK_U8X3(HE, PMK)                                                                                    \
    warp_t_u8x3<HE, PMK><<<grid, 256, 0, st>>>((const uint8_t*)payload, flow, sign, pmask, fmask, (uint8_t*)out, \
                                               omask, rule, H, W, packed)
    const bool pmk = pmask != nullptr && omask != nullptr;
    if (half_even && pmk) OFK_U8X3(true, true);
    else if (half_even) OFK_U8X3(true, false);
    else if (pmk) OFK_U8X3(false, true);
    else OFK_U8X3(false, false);
#undef OFK_U8X3
    OFK_LAUNCHED();
    return OFK_OK;
}

template <typename T, int AR>
static int launch_generic(const void* payload, int C, const float* flow, float sign, const uint8_t* pmask,
                          const uint8_t* fmask, void* out, uint8_t* omask, int rule, int N, int H, int W, int Hs,
                          int Ws, int Ho, int Wo, int oy, int ox, int fy, int fx, cudaStream_t st) {
    dim3 grid((Wo + 31) / 32, (Ho + 7) / 8, N);
    warp_t_generic<T, AR><<<grid, 256, 0, st>>>(static_cast<const T*>(payload), C, flow, sign, pmask, fmask,
                                                static_cast<T*>(out), omask, rule, H, W, Hs, Ws, Ho, Wo, oy, ox, fy,
                                                fx);
    OFK_LAUNCHED();
    return OFK_OK;
}

// warp_t_ws.cu
int launch_warp_u8_ws(int C, bool half_even, const void* payload, const float* flow, float sign, const uint8_t* pmask,
                      const uint8_t* fmask, void* out, uint8_t* omask, int rule, int N, int H, int W, cudaStream_t st);
bool warp_ws_enabled();
// combine3_ws.cu
int launch_combine3_ws(const float* P, const uint8_t* Pm, const float* G, const uint8_t* Gm, float sign, bool add,
                       float* out, uint8_t* omask, int N, int H, int W, cudaStream_t st);
bool c3_ws_enabled();

}  // namespace ofk

using namespace ofk;

extern "C" int ofk_warp_t(const void* payload, int dtype, int C, int arith, const float* flow, float flow_sign,
                          const uint8_t* payload_mask, const uint8_t* flow_mask, void* out, uint8_t* out_mask,
                          int mask_rule, int N, int H, int W, int Hs, int Ws, int top, int left, int cut,
                          ofk_stream_t stream) {
    OFK_CHECK_ARG(flow != nullptr, "ofk_warp_t: flow is NULL");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0 && Hs > 0 && Ws > 0, "ofk_warp_t: bad shape N=%d H=%d W=%d Hs=%d Ws=%d", N,
                  H, W, Hs, Ws);
    OFK_CHECK_ARG(C >= 0 && (C == 0 || (payload != nullptr && out != nullptr)),
                  "ofk_warp_t: payload/out NULL with C=%d", C);
    OFK_CHECK_ARG(C > 0 || out_mask != nullptr, "ofk_warp_t: nothing to compute (C=0 and out_mask NULL)");
    OFK_CHECK_ARG(dtype >= OFK_U8 && dtype <= OFK_F64, "ofk_warp_t: unknown dtype %d", dtype);
    OFK_CHECK_ARG(mask_rule >= OFK_RULE_STRICT && mask_rule <= OFK_RULE_GE_HALF, "ofk_warp_t: unknown mask rule %d",
                  mask_rule);
    OFK_CHECK_ARG(top >= 0 && left >= 0 && top + H <= Hs && left + W <= Ws,
                  "ofk_warp_t: flow frame (%d,%d)+(%d,%d) does not fit the payload frame (%d,%d)", top, left, H, W, Hs,
                  Ws);
    OFK_CHECK_ARG(flow_sign == 1.0f || flow_sign == -1.0f, "ofk_warp_t: flow_sign must be +1 or -1");
    if (N == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_warp_t: N=%d exceeds 65535 frames per call", N);
    cudaStream_t st = as_stream(stream);

    const bool same_frame = (Hs == H && Ws == W);
    struct PathCount {   // every exit below that is not a TMA launch is a gather-kernel launch
        bool tma = false;
        ~PathCount() { g_paths[tma ? 2 : 3].fetch_add(1, std::memory_order_relaxed); }
    } path;
    int ar;
    switch (dtype) {
        case OFK_U8: ar = (arith == OFK_ARITH_RINT) ? AR_RINT : AR_U8_FIXED; break;
        case OFK_I16:
        case OFK_U16: ar = AR_RINT; break;
        case OFK_F32: ar = AR_F32; break;
        default: ar = AR_F64; break;
    }
    // rows kernels: same frame for flow and payload, natural alignment, frame-local 32-bit offsets
    const bool fast = same_frame && H < 32768 && W < 32768 && ((size_t)H * W * (C > 0 ? C : 1) < (size_t)1 << 30) &&
                      ((reinterpret_cast<uintptr_t>(flow) & 7) == 0) &&
                      (C == 0 || (aligned16(payload) && aligned16(out)));
    if (fast) {
#define OFK_ROWS(T, CC, AR) \
    return launch_rows<T, CC, AR>(payload, flow, flow_sign, payload_mask, flow_mask, out, out_mask, mask_rule, N, H, W, st)
        if (C == 0) OFK_ROWS(uint8_t, 0, AR_U8_FIXED);
        // a flow warped by a flow (Flow.apply(Flow), 27 B/px): the composition kernel without its addition
        if (dtype == OFK_F32 && C == 2 && out_mask != nullptr && mask_rule == OFK_RULE_STRICT && c3_ws_enabled() &&
            ((payload_mask == nullptr) == (flow_mask == nullptr)) && aligned16(flow) && aligned16(out_mask) &&
            aligned16(payload_mask) && aligned16(flow_mask)) {
            const int ws = launch_combine3_ws(flow, flow_mask, static_cast<const float*>(payload), payload_mask, flow_sign,
                                              false, static_cast<float*>(out), out_mask, N, H, W, st);
            path.tma = ws > 0;
            if (ws != 0) return ws < 0 ? ws : OFK_OK;
        }
        if (dtype == OFK_U8 && (C == 1 || C == 3 || C == 4) && warp_ws_enabled()) {
            const int ws = launch_warp_u8_ws(C, ar == AR_RINT, payload, flow, flow_sign, payload_mask, flow_mask, out,
                                             out_mask, mask_rule, N, H, W, st);
            path.tma = ws > 0;
            if (ws != 0) return ws < 0 ? ws : OFK_OK;
        }
        if (dtype == OFK_U8 && C == 3)
            return launch_u8x3(ar == AR_RINT, payload, flow, flow_sign, payload_mask, flow_mask, out, out_mask,
                               mask_rule, N, H, W, st);
        if (dtype == OFK_U8 && ar == AR_U8_FIXED) {
            if (C == 1) OFK_ROWS(uint8_t, 1, AR_U8_FIXED);
            if (C == 4) OFK_ROWS(uint8_t, 4, AR_U8_FIXED);
        } else if (dtype == OFK_U8 && ar == AR_RINT) {
            if (C == 1) OFK_ROWS(uint8_t, 1, AR_RINT);
            if (C == 4) OFK_ROWS(uint8_t, 4, AR_RINT);
        } else if (dtype == OFK_F32) {
            if (C == 2) OFK_ROWS(float, 2, AR_F32);
            if (C == 3) OFK_ROWS(float, 3, AR_F32);
            if (C == 1) OFK_ROWS(float, 1, AR_F32);
            if (C == 4) OFK_ROWS(float, 4, AR_F32);
        }
#undef OFK_ROWS
    }
    // generic path: output frame is the flow frame (cut) or the payload frame (no cut)
    const int Ho = cut ? H : Hs, Wo = cut ? W : Ws;
    const int oy = cut ? top : 0, ox = cut ? left : 0;
    const int fy = cut ? 0 : top, fx = cut ? 0 : left;
#define OFK_GEN(T, AR)                                                                                              \
    return launch_generic<T, AR>(payload, C, flow, flow_sign, payload_mask, flow_mask, out, out_mask, mask_rule, N, H, \
                                 W, Hs, Ws, Ho, Wo, oy, ox, fy, fx, st)
    switch (dtype) {
        case OFK_U8:
            if (ar == AR_RINT) OFK_GEN(uint8_t, AR_RINT);
            OFK_GEN(uint8_t, AR_U8_FIXED);
        case OFK_I16: OFK_GEN(int16_t, AR_RINT);
        case OFK_U16: OFK_GEN(uint16_t, AR_RINT);
        case OFK_F32: OFK_GEN(float, AR_F32);
        default: OFK_GEN(double, AR_F64);
    }
#undef OFK_GEN
}

extern "C" int ofk_warp_t_ex(const void* payload, int dtype, int C, int arith, const float* flow, float flow_sign,
                             const uint8_t* payload_mask, const uint8_t* flow_mask, const int* flow_nonzero, void* out,
                             uint8_t* out_mask, int mask_rule, int N, int H, int W, int Hs, int Ws, int top, int left,
                             int cut, ofk_stream_t stream) {
    const int rc = ofk_warp_t(payload, dtype, C, arith, flow, flow_sign, payload_mask, flow_mask, out, out_mask,
                              mask_rule, N, H, W, Hs, Ws, top, left, cut, stream);
    if (rc != OFK_OK || flow_nonzero == nullptr || C == 0 || N == 0) return rc;
    const int Ho = cut ? H : Hs;
    const long long rowlen = (long long)(cut ? W : Ws) * C, src_row = (long long)Ws * C;
    const long long src_off = cut ? (long long)top * src_row + (long long)left * C : 0;
    dim3 grid((unsigned)std::min<long long>((rowlen + 255) / 256, 8), (unsigned)std::min(Ho, 64), N);
    cudaStream_t st = as_stream(stream);
#define OFK_PASS(E)                                                                                                \
    warp_t_passthrough<E><<<grid, 256, 0, st>>>(static_cast<const E*>(payload), flow_nonzero, static_cast<E*>(out), \
                                                Ho, rowlen, src_row, src_off, (long long)Hs * src_row)
    switch (dtype) {
        case OFK_U8: OFK_PASS(uint8_t); break;
        case OFK_I16:
        case OFK_U16: OFK_PASS(uint16_t); break;
        case OFK_F32: OFK_PASS(uint32_t); break;
        default: OFK_PASS(unsigned long long); break;
    }
#undef OFK_PASS
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_valid_geom_t(const float* flow, float flow_sign, const uint8_t* flow_mask, uint8_t* out, int N,
                                int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(out != nullptr, "ofk_valid_geom_t: out is NULL");
    OFK_CHECK_ARG(flow != nullptr && N >= 0 && H > 0 && W > 0, "ofk_valid_geom_t: bad arguments");
    OFK_CHECK_ARG(flow_sign == 1.0f || flow_sign == -1.0f, "ofk_valid_geom_t: flow_sign must be +1 or -1");
    if (N == 0) return OFK_OK;
    if (W % 4 == 0 && W < 32768 && H < 32768 && aligned16(flow) && (reinterpret_cast<uintptr_t>(out) & 3) == 0 &&
        (reinterpret_cast<uintptr_t>(flow_mask) & 3) == 0) {
        const size_t qpf = (size_t)H * W / 4;
        if (qpf < 0x7fffff00ull && N <= 65535) {
            valid_geom_vec4<<<dim3((unsigned)((qpf + 255) / 256), N), 256, 0, as_stream(stream)>>>(
                reinterpret_cast<const float4*>(flow), flow_sign, reinterpret_cast<const uint32_t*>(flow_mask),
                reinterpret_cast<uint32_t*>(out), H, W, (unsigned)qpf);
            OFK_LAUNCHED();
            return OFK_OK;
        }
    }
    return ofk_warp_t(nullptr, OFK_U8, 0, OFK_ARITH_NATIVE, flow, flow_sign, nullptr, flow_mask, nullptr, out,
                      OFK_RULE_STRICT, N, H, W, H, W, 0, 0, 1, stream);
}
