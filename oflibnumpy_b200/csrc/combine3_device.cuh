// Device helpers shared by the composition kernels (combine3.cu, tma_kernels.cu). Everything is static so each
// translation unit gets its own copy (the library is built without relocatable device code).
#pragma once
#include "ofk_common.cuh"

namespace ofk {

// Epilogues of the sampling kernels (c3_ws_kernel, combine3_rows): what a pixel writes once s = Q(G, p + sign*P[p])
// and its validity (P mask & strict G mask at the taps) are known.
constexpr int EPI_SAMPLE = 0;    // out = s, mask = valid                    (Flow.apply of a flow, ofk_warp_t)
constexpr int EPI_COMPOSE = 1;   // out = P + s, mask = valid                (ofk_combine3)
constexpr int EPI_CONSIST = 2;   // out = valid & fb_consistent(P, s), one byte; optionally valid (ofk_consistency)

// Kernel arguments of an epilogue: none for sample and compose, so that their kernels keep their code.
template <int EPI>
struct EpiArgs {};
template <>
struct EpiArgs<EPI_CONSIST> {
    float a1, a2;
    uint8_t* valid;   // NULL: the valid byte is not written
};

// Forward-backward consistency (Sundaram, Brox & Keutzer, ECCV 2010) of w = P[p] and the sampled backward flow s:
//   |w + s|^2 < a1 (|w|^2 + |s|^2) + a2
// in float32, every operation rounded on its own (no FMA contraction), in this order.
__device__ __forceinline__ unsigned fb_consistent(float wu, float wv, float su, float sv, float a1, float a2) {
    const float ru = __fadd_rn(wu, su), rv = __fadd_rn(wv, sv);
    const float lhs = __fadd_rn(__fmul_rn(ru, ru), __fmul_rn(rv, rv));
    const float ww = __fadd_rn(__fmul_rn(wu, wu), __fmul_rn(wv, wv));
    const float ss = __fadd_rn(__fmul_rn(su, su), __fmul_rn(sv, sv));
    const float rhs = __fadd_rn(__fmul_rn(a1, __fadd_rn(ww, ss)), a2);
    return lhs < rhs ? 1u : 0u;
}

struct SampleResult {
    float u, v;
    int strict;
};

// exact but slow: any coordinates, taps may leave the frame (out of line, by-value in / out: no stack traffic)
static __device__ __noinline__ SampleResult sample_flow_border(const float2* __restrict__ G, const uint8_t* __restrict__ Gm,
                                                        int H, int W, float X, float Y) {
    const QCoord qx = quantise(X), qy = quantise(Y);
    const int ix = qx.i, iy = qy.i;
    const QWeights w = qweights(qx.f, qy.f);
    const bool x0 = (unsigned)ix < (unsigned)W, x1 = (unsigned)(ix + 1) < (unsigned)W;
    const bool y0 = (unsigned)iy < (unsigned)H, y1 = (unsigned)(iy + 1) < (unsigned)H;
    const long long o = (long long)iy * W + ix;
    const float2 z = make_float2(0.f, 0.f);
    const float2 t00 = (x0 && y0) ? __ldg(G + o) : z;
    const float2 t01 = (x1 && y0) ? __ldg(G + o + 1) : z;
    const float2 t10 = (x0 && y1) ? __ldg(G + o + W) : z;
    const float2 t11 = (x1 && y1) ? __ldg(G + o + W + 1) : z;
    int S = 0;
    if (x0 && y0 && (!Gm || __ldg(Gm + o))) S += w.w00;
    if (x1 && y0 && (!Gm || __ldg(Gm + o + 1))) S += w.w01;
    if (x0 && y1 && (!Gm || __ldg(Gm + o + W))) S += w.w10;
    if (x1 && y1 && (!Gm || __ldg(Gm + o + W + 1))) S += w.w11;
    const float s = 1.0f / 1024.0f;
    const float f00 = float(w.w00) * s, f01 = float(w.w01) * s, f10 = float(w.w10) * s, f11 = float(w.w11) * s;
    SampleResult r;
    r.u = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t00.x, f00), __fmul_rn(t01.x, f01)), __fmul_rn(t10.x, f10)),
                    __fmul_rn(t11.x, f11));
    r.v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t00.y, f00), __fmul_rn(t01.y, f01)), __fmul_rn(t10.y, f10)),
                    __fmul_rn(t11.y, f11));
    r.strict = (S == 1024);
    return r;
}

}  // namespace ofk
