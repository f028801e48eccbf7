// Fused flow composition, mode 3 (flow_class.py:1411-1422 of the reference) for sm_100a.
//
//   ref 't' : out[p] = B[p] + Q(A, p - B[p]);   out_mask[p] = Bm[p] & strict(Am at the taps)
//   ref 's' : out[p] = A[p] + Q(B, p + A[p]);   out_mask[p] = Am[p] & strict(Bm at the taps)
//
// Q is the cv2.remap float32 bilinear sample (1/32-px coordinates, zero border). The reference evaluates this as
// warp (remap of vecs||mask) -> Flow construction -> add -> mask AND, i.e. five full-frame passes plus two masked
// zero tests; here one kernel reads both operands once (27 B/px algorithmic) and also produces the zero-test flags
// that gate the reference's early exits (flow_class.py:1338-1354), which a second tiny kernel applies on the device.
#include <float.h>
#include <stdlib.h>

#include "combine3_device.cuh"

namespace ofk {

// "P" is the operand read at p (pointwise), "G" the operand gathered at p + sign*P[p].
__device__ __forceinline__ bool nonzero(float c, float thr) { return thr > 0.f ? !(c < thr && c > -thr) : (c != 0.f); }

// flags[n*2 + 0] = A has a non-zero vector on a valid pixel, flags[n*2 + 1] = same for B. Warps record what they saw
// in shared memory; the last warp of the CTA to finish publishes (no CTA-wide barrier at the tail, so finished warps
// release their slots immediately).
struct FlagScratch {
    int nzA, nzB, done;
};
__device__ __forceinline__ void publish_flags(bool nzA, bool nzB, int* __restrict__ flags, int n, FlagScratch* sc) {
    const bool a = __any_sync(0xffffffffu, nzA), b = __any_sync(0xffffffffu, nzB);
    if ((threadIdx.x & 31) == 0) {
        if (a) sc->nzA = 1;   // benign race: every writer stores the same value
        if (b) sc->nzB = 1;
        __threadfence_block();
        if (atomicAdd(&sc->done, 1) == (int)(blockDim.x >> 5) - 1) {
            __threadfence_block();
            if (*(volatile int*)&sc->nzA) flags[n * 2 + 0] = 1;
            if (*(volatile int*)&sc->nzB) flags[n * 2 + 1] = 1;
        }
    }
}

// Persistent kernel. CTA (bx, by) owns tile column bx (32 pixels wide, so x, its float and the column predicates are
// loop invariants of a thread) and walks over the 32-row tiles r = by, by + gridDim.y, ... of all frames stacked on top
// of each other; frame / tile-row are tracked incrementally (no divisions). In a tile a warp owns 32 consecutive
// pixels of a row (lane = x) and 4 rows, so every access of a warp instruction is contiguous along x: the pointwise
// operand, the zero-test read of the gathered operand and the output are fully coalesced, and each gather
// instruction touches the 2-3 cache lines of a rotated row segment.
// Latency is hidden in two ways: (1) the coalesced inputs of the NEXT tile are loaded into a second register set
// before the current tile is processed (software pipelining across tiles, no CTA churn); (2) inside a tile all
// gathers of all rows are issued before the first use. Tiles cut by the frame border take a clamped / predicated
// copy of the same code (FULL = false).
// REF_T: pointwise operand is B, gathered is A (sign -1); otherwise pointwise A, gathered B (sign +1).
struct TileIn {
    float2 p[4], g[4];
    unsigned pmv[4], gmv[4];
};

template <bool MASKS, bool FULL>
__device__ __forceinline__ void load_tile(TileIn& in, const float2* __restrict__ P, const float2* __restrict__ G,
                                          const uint8_t* __restrict__ Pm, const uint8_t* __restrict__ Gm,
                                          unsigned x, unsigned y0, int H, int W) {
    const unsigned xc = FULL ? x : min(x, (unsigned)W - 1);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned yc = FULL ? y0 + j : min(y0 + j, (unsigned)H - 1);
        const unsigned idx = yc * (unsigned)W + xc;
        in.p[j] = ld_stream_f2(P + idx);
        in.g[j] = __ldg(G + idx);         // zero test of the gathered operand AT p; these lines are gathered anyway
        in.pmv[j] = MASKS ? Pm[idx] : 1u;
        in.gmv[j] = MASKS ? __ldg(Gm + idx) : 1u;
    }
}

// EPI (combine3_device.cuh): EPI_COMPOSE writes O and Om; EPI_CONSIST writes the consistency byte to Om and, if Ov
// is not NULL, the valid byte to Ov (O is not used).
template <bool REF_T, bool MASKS, bool FULL, int EPI = EPI_COMPOSE>
__device__ __forceinline__ void process_tile(const TileIn& cur, const float2* __restrict__ G,
                                             const uint8_t* __restrict__ Gm, float2* __restrict__ O,
                                             uint8_t* __restrict__ Om, unsigned x, float Xg, unsigned y0, float tz,
                                             int H, int W, unsigned& nzP, unsigned& nzG,
                                             const EpiArgs<EPI>& epi = EpiArgs<EPI>{},
                                             uint8_t* __restrict__ Ov = nullptr) {
    const float sign = REF_T ? -1.0f : 1.0f;
    // phase 1: zero tests and quantised sample coordinates of all rows (no control flow)
    float X[4], Y[4];
    QCoord qx[4], qy[4];
    bool interior = true;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        nzP |= cur.pmv[j] & (unsigned)(fabsf(cur.p[j].x) >= tz || fabsf(cur.p[j].y) >= tz);
        nzG |= cur.gmv[j] & (unsigned)(fabsf(cur.g[j].x) >= tz || fabsf(cur.g[j].y) >= tz);
        X[j] = __fmaf_rn(sign, cur.p[j].x, Xg);
        Y[j] = __fmaf_rn(sign, cur.p[j].y, static_cast<float>(y0 + j));
        qx[j] = quantise_fast(X[j]);
        qy[j] = quantise_fast(Y[j]);
        interior = interior && (unsigned)qx[j].i < (unsigned)(W - 1) && (unsigned)qy[j].i < (unsigned)(H - 1) &&
                   fabsf(X[j]) < OFK_FAST_COORD_LIMIT && fabsf(Y[j]) < OFK_FAST_COORD_LIMIT;
    }
    float su[4], sv[4];
    unsigned strict[4];
    if (__all_sync(0xffffffffu, interior)) {
        // phase 2 (whole warp interior, the common case): every gather of every row before the first use
        float2 tp[4][4];
        unsigned inv[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const unsigned o = (unsigned)(qy[j].i * W + qx[j].i);
            const float2* g0 = G + o;
            const float2* g1 = g0 + W;
            tp[j][0] = __ldg(g0); tp[j][1] = __ldg(g0 + 1); tp[j][2] = __ldg(g1); tp[j][3] = __ldg(g1 + 1);
            if (MASKS) {
                const uint8_t* m0 = Gm + o;
                const uint8_t* m1 = m0 + W;
                inv[j][0] = __ldg(m0); inv[j][1] = __ldg(m0 + 1); inv[j][2] = __ldg(m1); inv[j][3] = __ldg(m1 + 1);
            }
        }
        // phase 3: blend in cv2.remap's order (left to right, no FMA contraction)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int a = qx[j].f, b = qy[j].f;
            strict[j] = 1;
            if (MASKS) {
                // a tap only matters when its weight is non-zero: (32-a)(32-b), a(32-b), (32-a)b, ab
                const unsigned za = a == 0, zb = b == 0;
                strict[j] = inv[j][0] & (inv[j][1] | za) & (inv[j][2] | zb) & (inv[j][3] | za | zb);
            }
            const float fa = (float)a * (1.0f / 32.0f), fb = (float)b * (1.0f / 32.0f);
            const float na = 1.0f - fa, nb = 1.0f - fb;                  // exact: multiples of 1/32
            const float f00 = __fmul_rn(na, nb), f01 = __fmul_rn(fa, nb), f10 = __fmul_rn(na, fb),
                        f11 = __fmul_rn(fa, fb);
            su[j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(tp[j][0].x, f00), __fmul_rn(tp[j][1].x, f01)),
                                        __fmul_rn(tp[j][2].x, f10)), __fmul_rn(tp[j][3].x, f11));
            sv[j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(tp[j][0].y, f00), __fmul_rn(tp[j][1].y, f01)),
                                        __fmul_rn(tp[j][2].y, f10)), __fmul_rn(tp[j][3].y, f11));
        }
    } else {
        // some tap of this warp touches the border (or leaves the fast quantiser's range): exact per-pixel path
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const SampleResult r = sample_flow_border(G, MASKS ? Gm : nullptr, H, W, X[j], Y[j]);
            su[j] = r.u; sv[j] = r.v; strict[j] = (unsigned)r.strict;
        }
    }
    if (FULL || x < (unsigned)W) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const unsigned y = y0 + j;
            if (FULL || y < (unsigned)H) {
                const unsigned idx = y * (unsigned)W + x;
                if constexpr (EPI == EPI_CONSIST) {
                    const unsigned v = cur.pmv[j] & strict[j];
                    Om[idx] = (uint8_t)(v & fb_consistent(cur.p[j].x, cur.p[j].y, su[j], sv[j], epi.a1, epi.a2));
                    if (Ov != nullptr) Ov[idx] = (uint8_t)v;
                } else {
                    float2 o;
                    o.x = __fadd_rn(cur.p[j].x, su[j]);
                    o.y = __fadd_rn(cur.p[j].y, sv[j]);
                    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(O + idx), "f"(o.x), "f"(o.y)
                                 : "memory");
                    Om[idx] = (uint8_t)(cur.pmv[j] & strict[j]);
                }
            }
        }
    }
}

// Linear tile index -> (frame, tile row, tile column), advanced incrementally by the grid stride (no divisions).
struct TileIter {
    int n, ty, tx;      // current tile
    int dn, dy, dx;     // grid stride decomposed in the same mixed radix
    __device__ __forceinline__ void init(unsigned t, unsigned stride, int tiles_x, int tiles_y) {
        const unsigned per_frame = (unsigned)tiles_x * tiles_y;
        n = t / per_frame;
        unsigned r = t - n * per_frame;
        ty = r / tiles_x;
        tx = r - ty * tiles_x;
        dn = stride / per_frame;
        r = stride - dn * per_frame;
        dy = r / tiles_x;
        dx = r - dy * tiles_x;
    }
    __device__ __forceinline__ void advance(int tiles_x, int tiles_y) {
        tx += dx;
        if (tx >= tiles_x) { tx -= tiles_x; ++ty; }
        ty += dy;
        if (ty >= tiles_y) { ty -= tiles_y; ++n; }
        n += dn;
    }
};

// EPI_CONSIST (ofk_consistency): omask receives the consistency byte, epi.valid (if set) the valid byte; out is not
// used and flags must be NULL.
template <bool REF_T, bool MASKS, int MINB, int EPI = EPI_COMPOSE>
__global__ void __launch_bounds__(256, MINB) combine3_rows(const float* __restrict__ A, const uint8_t* __restrict__ Am,
                                                           const float* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                           float thr, float* __restrict__ out,
                                                           uint8_t* __restrict__ omask, int* __restrict__ flags, int H,
                                                           int W, int tiles_x, int tiles_y, int N,
                                                           const EpiArgs<EPI> epi = EpiArgs<EPI>{}) {
    // zero test as one compare per component: |c| >= t with t = thr, or the smallest denormal for the exact test
    const float tz = thr > 0.f ? thr : 1.401298464e-45f;
    const unsigned lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const size_t frame = (size_t)H * W;
    TileIter it;
    it.init(blockIdx.x, gridDim.x, tiles_x, tiles_y);
    if (it.n >= N) return;
    const float2* Pb = reinterpret_cast<const float2*>(REF_T ? B : A);
    const float2* Gb = reinterpret_cast<const float2*>(REF_T ? A : B);
    const uint8_t* Pmb = MASKS ? (REF_T ? Bm : Am) : nullptr;
    const uint8_t* Gmb = MASKS ? (REF_T ? Am : Bm) : nullptr;

    TileIn cur;
    {
        const size_t fb = (size_t)it.n * frame;
        load_tile<MASKS, false>(cur, Pb + fb, Gb + fb, Pmb + fb, Gmb + fb, (unsigned)it.tx * 32 + lane,
                                (unsigned)it.ty * 32 + wrp * 4, H, W);
    }
    unsigned nzP = 0, nzG = 0;
    for (;;) {
        const int n = it.n;
        const size_t fbase = (size_t)n * frame;
        const unsigned x = (unsigned)it.tx * 32 + lane, y0 = (unsigned)it.ty * 32 + wrp * 4;
        const bool full = (it.tx * 32 + 32 <= W) && (it.ty * 32 + 32 <= H);
        it.advance(tiles_x, tiles_y);
        const bool more = it.n < N;
        TileIn nxt = cur;
        if (more) {   // block-uniform; clamped loads so that partial tiles can be prefetched too
            const size_t fb2 = (size_t)it.n * frame;
            load_tile<MASKS, false>(nxt, Pb + fb2, Gb + fb2, Pmb + fb2, Gmb + fb2, (unsigned)it.tx * 32 + lane,
                                    (unsigned)it.ty * 32 + wrp * 4, H, W);
        }
        if constexpr (EPI == EPI_CONSIST) {
            uint8_t* Om = omask + fbase;
            uint8_t* Ov = epi.valid != nullptr ? epi.valid + fbase : nullptr;
            const float Xg = static_cast<float>(x);
            if (full)
                process_tile<REF_T, MASKS, true, EPI>(cur, Gb + fbase, Gmb + fbase, nullptr, Om, x, Xg, y0, tz, H, W, nzP,
                                                      nzG, epi, Ov);
            else
                process_tile<REF_T, MASKS, false, EPI>(cur, Gb + fbase, Gmb + fbase, nullptr, Om, x, Xg, y0, tz, H, W,
                                                       nzP, nzG, epi, Ov);
        } else {
            float2* O = reinterpret_cast<float2*>(out) + fbase;
            uint8_t* Om = omask + fbase;
            const float Xg = static_cast<float>(x);
            if (full)
                process_tile<REF_T, MASKS, true>(cur, Gb + fbase, Gmb + fbase, O, Om, x, Xg, y0, tz, H, W, nzP, nzG);
            else
                process_tile<REF_T, MASKS, false>(cur, Gb + fbase, Gmb + fbase, O, Om, x, Xg, y0, tz, H, W, nzP, nzG);
        }
        // publish the zero-test result when this CTA leaves the frame (clamped duplicates of partial tiles repeat
        // pixels of the same frame, so they cannot create false positives)
        if (flags != nullptr && (!more || it.n != n)) {
            const bool fa_ = __any_sync(0xffffffffu, (REF_T ? nzG : nzP) != 0);
            const bool fb_ = __any_sync(0xffffffffu, (REF_T ? nzP : nzG) != 0);
            if (lane == 0) {
                if (fa_) flags[n * 2 + 0] = 1;   // benign race: every writer stores the same value
                if (fb_) flags[n * 2 + 1] = 1;
            }
            nzP = 0;
            nzG = 0;
        }
        if (!more) break;
        cur = nxt;
    }
}

__device__ __forceinline__ void publish_flags_barrier(bool nzA, bool nzB, int* __restrict__ flags, int n) {
    const int a = __syncthreads_or(nzA);
    const int b = __syncthreads_or(nzB);
    if (threadIdx.x == 0) {
        if (a) flags[n * 2 + 0] = 1;
        if (b) flags[n * 2 + 1] = 1;
    }
}

// scalar fallback: any W, any alignment
template <bool REF_T>
__global__ void __launch_bounds__(256) combine3_scalar(const float* __restrict__ A, const uint8_t* __restrict__ Am,
                                                       const float* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                       float thr, float* __restrict__ out,
                                                       uint8_t* __restrict__ omask, int* __restrict__ flags, int H,
                                                       int W) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int n = blockIdx.z;
    const size_t frame = (size_t)H * W;
    bool nzP = false, nzG = false;
    if (x < W && y < H) {
        const size_t pix = (size_t)n * frame + (size_t)y * W + x;
        const float* P = REF_T ? B : A;
        const uint8_t* Pm = REF_T ? Bm : Am;
        const float* G = REF_T ? A : B;
        const uint8_t* Gm = REF_T ? Am : Bm;
        const float sign = REF_T ? -1.0f : 1.0f;
        const float pu = P[pix * 2], pv = P[pix * 2 + 1];
        const float gu = G[pix * 2], gv = G[pix * 2 + 1];
        const bool pvalid = Pm ? Pm[pix] != 0 : true, gvalid = Gm ? Gm[pix] != 0 : true;
        nzP = pvalid && (nonzero(pu, thr) || nonzero(pv, thr));
        nzG = gvalid && (nonzero(gu, thr) || nonzero(gv, thr));
        const float X = __fadd_rn(sign * pu, static_cast<float>(x));
        const float Y = __fadd_rn(sign * pv, static_cast<float>(y));
        // float2 gathers need 8-byte alignment of the frame base; the scalar path cannot assume it
        const QCoord qx = quantise(X), qy = quantise(Y);
        const int ix = qx.i, iy = qy.i;
        const QWeights w = qweights(qx.f, qy.f);
        const bool x0 = (unsigned)ix < (unsigned)W, x1 = (unsigned)(ix + 1) < (unsigned)W;
        const bool y0 = (unsigned)iy < (unsigned)H, y1 = (unsigned)(iy + 1) < (unsigned)H;
        const float* Gf = G + (size_t)n * frame * 2;
        const uint8_t* Gmf = Gm ? Gm + (size_t)n * frame : nullptr;
        const long long o = (long long)iy * W + ix;
        const bool in[4] = {x0 && y0, x1 && y0, x0 && y1, x1 && y1};
        const long long off[4] = {o, o + 1, o + W, o + W + 1};
        const int wi[4] = {w.w00, w.w01, w.w10, w.w11};
        float au = 0.f, av = 0.f;
        int S = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float tu = in[k] ? Gf[off[k] * 2] : 0.f, tv = in[k] ? Gf[off[k] * 2 + 1] : 0.f;
            const float f = float(wi[k]) * (1.0f / 1024.0f);
            au = (k == 0) ? __fmul_rn(tu, f) : __fadd_rn(au, __fmul_rn(tu, f));
            av = (k == 0) ? __fmul_rn(tv, f) : __fadd_rn(av, __fmul_rn(tv, f));
            if (in[k] && (Gmf == nullptr || Gmf[off[k]])) S += wi[k];
        }
        out[pix * 2] = __fadd_rn(pu, au);
        out[pix * 2 + 1] = __fadd_rn(pv, av);
        omask[pix] = (pvalid && S == 1024) ? 1 : 0;
    }
    if (flags != nullptr) publish_flags_barrier(REF_T ? nzG : nzP, REF_T ? nzP : nzG, flags, n);
}

// Early exits of combine_with (flow_class.py:1338-1354), applied on the device: frame n becomes a copy of B when A
// is zero on its valid pixels, else a copy of A when B is. A NULL input mask means all valid (copied as ones).
__global__ void __launch_bounds__(256) combine3_fixup(const float* __restrict__ A, const uint8_t* __restrict__ Am,
                                                      const float* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                      const int* __restrict__ flags, float* __restrict__ out,
                                                      uint8_t* __restrict__ omask, size_t frame) {
    const int n = blockIdx.y;
    const int a_nz = flags[n * 2], b_nz = flags[n * 2 + 1];
    if (a_nz && b_nz) return;
    const float* src = a_nz ? A : B;  // A zero -> B wins (tested first, like the reference); else B zero -> A
    const uint8_t* srcm = a_nz ? Am : Bm;
    const size_t base = (size_t)n * frame;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < frame; i += (size_t)gridDim.x * blockDim.x) {
        out[(base + i) * 2] = src[(base + i) * 2];
        out[(base + i) * 2 + 1] = src[(base + i) * 2 + 1];
        omask[base + i] = srcm ? srcm[base + i] : 1;
    }
}

}  // namespace ofk

namespace ofk {   // combine3_ws.cu
int launch_combine3_ws(const float* P, const uint8_t* Pm, const float* G, const uint8_t* Gm, float sign, bool add,
                       float* out, uint8_t* omask, int N, int H, int W, cudaStream_t st);
int launch_c3_zero_flags(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float thr, int* flags,
                         int N, int H, int W, cudaStream_t st);
int launch_consistency_ws(const float* F, const uint8_t* Fm, const float* G, const uint8_t* Gm, float sign, float a1,
                          float a2, uint8_t* out, uint8_t* out_valid, int N, int H, int W, cudaStream_t st);
bool c3_ws_enabled();
}

using namespace ofk;

extern "C" int ofk_combine3(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, int ref, float thr,
                            float* out, uint8_t* out_mask, int* flags, int N, int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(A && B && out && out_mask, "ofk_combine3: NULL operand (A=%p B=%p out=%p out_mask=%p)", (void*)A,
                  (void*)B, (void*)out, (void*)out_mask);
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofk_combine3: ref must be 's' or 't', got %d", ref);
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0, "ofk_combine3: bad shape N=%d H=%d W=%d", N, H, W);
    OFK_CHECK_ARG(thr >= 0.f, "ofk_combine3: negative threshold");
    if (N == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_combine3: N=%d exceeds 65535 frames per call", N);
    OFK_CHECK_ARG((double)N * ((H + 31) / 32) * ((W + 31) / 32) < 2.0e9, "ofk_combine3: too many tiles");
    cudaStream_t st = as_stream(stream);
    const bool fast = ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) |
                        reinterpret_cast<uintptr_t>(out)) & 7) == 0 && (size_t)H * W < ((size_t)1 << 30) && H < 32768 &&
                      W < 32768 && ((Am == nullptr) == (Bm == nullptr));
    // default: the warp-specialised TMA kernel (16-byte aligned frames, W % 16 == 0); its zero tests are separate
    // launches. Everything else: the register-pipelined gather kernel, which tests for zero on the fly.
    int ws = 0;
    if (fast && c3_ws_enabled() && ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B) |
                                     reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(out_mask) |
                                     reinterpret_cast<uintptr_t>(Am) | reinterpret_cast<uintptr_t>(Bm)) & 15) == 0) {
        if (ref == 't') ws = launch_combine3_ws(B, Bm, A, Am, -1.0f, true, out, out_mask, N, H, W, st);
        else ws = launch_combine3_ws(A, Am, B, Bm, 1.0f, true, out, out_mask, N, H, W, st);
        if (ws < 0) return ws;
        if (ws == 1 && flags != nullptr) {
            const int rc = launch_c3_zero_flags(A, Am, B, Bm, thr, flags, N, H, W, st);
            if (rc != OFK_OK) return rc;
        }
    }
    if (ws != 1 && flags != nullptr) OFK_CUDA(cudaMemsetAsync(flags, 0, sizeof(int) * 2 * (size_t)N, st));
    g_paths[ws == 1 ? 0 : 1].fetch_add(1, std::memory_order_relaxed);
    if (ws == 1) {
        // launched
    } else if (fast) {
        static int variant = -1;
        if (variant < 0) {
            const char* e = getenv("OFK_C3_VARIANT");
            variant = e ? atoi(e) : 0;
        }
        const int tiles_x = (W + 31) / 32, tiles_y = (H + 31) / 32;
#define OFK_C3R(RT, MK, MINB, CPS)                                                                            \
    do {                                                                                                      \
        const long long total_ = (long long)tiles_x * tiles_y * N;                                            \
        long long grid_ = (long long)sm_count() * CPS; /* every CTA co-resident: no second wave */           \
        if (grid_ > total_) grid_ = total_;                                                                   \
        combine3_rows<RT, MK, MINB><<<(unsigned)grid_, 256, 0, st>>>(A, Am, B, Bm, thr, out, out_mask, flags, \
                                                                     H, W, tiles_x, tiles_y, N);              \
    } while (0)
#define OFK_C3V(MINB, CPS)                              \
    do {                                                \
        if (Am && Bm) {                                 \
            if (ref == 't') OFK_C3R(true, true, MINB, CPS);   \
            else OFK_C3R(false, true, MINB, CPS);             \
        } else {                                        \
            if (ref == 't') OFK_C3R(true, false, MINB, CPS);  \
            else OFK_C3R(false, false, MINB, CPS);            \
        }                                               \
    } while (0)
        switch (variant) {
            case 1: OFK_C3V(3, 3); break;
            case 2: OFK_C3V(4, 4); break;
            case 3: OFK_C3V(1, 1); break;
            default: OFK_C3V(2, 2); break;
        }
#undef OFK_C3V
#undef OFK_C3R
    } else {
        dim3 grid((W + 31) / 32, (H + 7) / 8, N);
        if (ref == 't') combine3_scalar<true><<<grid, 256, 0, st>>>(A, Am, B, Bm, thr, out, out_mask, flags, H, W);
        else combine3_scalar<false><<<grid, 256, 0, st>>>(A, Am, B, Bm, thr, out, out_mask, flags, H, W);
    }
    if (ws != 1) OFK_LAUNCHED();
    if (flags != nullptr) {
        const size_t frame = (size_t)H * W;
        int bx = (int)((frame + 256 * 8 - 1) / (256 * 8));
        if (bx > 64) bx = 64;
        combine3_fixup<<<dim3(bx, N), 256, 0, st>>>(A, Am, B, Bm, flags, out, out_mask, frame);
        OFK_LAUNCHED();
    }
    return OFK_OK;
}

// Forward-backward consistency of F (forward) and G (backward): one launch of the TMA kernel or of the rows kernel with
// the consistency epilogue; no zero tests, no early exits.
extern "C" int ofk_consistency(const float* F, const uint8_t* Fm, const float* G, const uint8_t* Gm, int ref,
                               float alpha1, float alpha2, uint8_t* out, uint8_t* out_valid, int N, int H, int W,
                               ofk_stream_t stream) {
    OFK_CHECK_ARG(F && G && out, "ofk_consistency: NULL pointer (F=%p G=%p out=%p)", (void*)F, (void*)G, (void*)out);
    OFK_CHECK_ARG((Fm == nullptr) == (Gm == nullptr), "ofk_consistency: Fm and Gm must both be given or both be NULL");
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofk_consistency: ref must be 's' or 't', got %d", ref);
    OFK_CHECK_ARG(alpha1 >= 0.f && alpha1 <= FLT_MAX && alpha2 >= 0.f && alpha2 <= FLT_MAX,
                  "ofk_consistency: alpha1 and alpha2 must be finite and >= 0 (alpha1=%g alpha2=%g)", (double)alpha1,
                  (double)alpha2);
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0 && H < 32768 && W < 32768 && (long long)H * W < (1ll << 30),
                  "ofk_consistency: bad shape N=%d H=%d W=%d (H and W below 32768, H*W below 2^30)", N, H, W);
    OFK_CHECK_ARG(N <= 65535, "ofk_consistency: N=%d exceeds 65535 frames per call", N);
    OFK_CHECK_ARG(((reinterpret_cast<uintptr_t>(F) | reinterpret_cast<uintptr_t>(G)) & 7) == 0,
                  "ofk_consistency: F and G must be 8-byte aligned (F=%p G=%p)", (void*)F, (void*)G);
    if (N == 0) return OFK_OK;
    cudaStream_t st = as_stream(stream);
    const float sign = ref == 't' ? -1.0f : 1.0f;
    // the TMA kernel where the tensor maps accept the operands (W % 16 == 0, 16-byte aligned), else the rows kernel
    int ws = 0;
    if (c3_ws_enabled()) {
        ws = launch_consistency_ws(F, Fm, G, Gm, sign, alpha1, alpha2, out, out_valid, N, H, W, st);
        if (ws < 0) return ws;
    }
    g_consistency_paths[ws == 1 ? 0 : 1].fetch_add(1, std::memory_order_relaxed);
    if (ws == 1) return OFK_OK;
    EpiArgs<EPI_CONSIST> epi;
    epi.a1 = alpha1;
    epi.a2 = alpha2;
    epi.valid = out_valid;
    const int tiles_x = (W + 31) / 32, tiles_y = (H + 31) / 32;
    long long grid = (long long)sm_count() * 2;   // every CTA co-resident, as the composition's default
    if (grid > (long long)tiles_x * tiles_y * N) grid = (long long)tiles_x * tiles_y * N;
    // combine3_rows reads P = B, G = A for REF_T, P = A, G = B otherwise: here P is always F
#define OFK_CONS(RT, MK)                                                                                          \
    combine3_rows<RT, MK, 2, EPI_CONSIST><<<(unsigned)grid, 256, 0, st>>>(RT ? G : F, RT ? Gm : Fm, RT ? F : G, \
                                                                          RT ? Fm : Gm, 0.f, nullptr, out,     \
                                                                          nullptr, H, W, tiles_x, tiles_y, N, epi)
    if (Fm != nullptr) {
        if (ref == 't') OFK_CONS(true, true);
        else OFK_CONS(false, true);
    } else {
        if (ref == 't') OFK_CONS(true, false);
        else OFK_CONS(false, false);
    }
#undef OFK_CONS
    OFK_LAUNCHED();
    return OFK_OK;
}
