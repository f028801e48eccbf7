// Accumulation of clips of flows to their keyframe, mode-3 composition folded over each clip (ofk_accumulate).
//
// A batch of S*L frames is S clips of L consecutive frames B_0 .. B_{L-1}. Mode 3 reads one operand at p and samples
// the other (combine3.cu), so both folds that can be walked are pointwise in the running flow:
//   ref 's' (left fold):  C_0 = B_0,      C_k = C_{k-1} (+) B_k:  C_k(p) = C_{k-1}(p) + Q(B_k, p + C_{k-1}(p))
//   ref 't' (right fold): D_{L-1} = B_{L-1}, D_j = B_j (+) D_{j+1}: D_j(p) = D_{j+1}(p) + Q(B_j, p - D_{j+1}(p))
// with the early exits of combine_with (self tested first): 's' C_{k-1} zero -> B_k, else B_k zero -> C_{k-1};
// 't' B_j zero -> D_{j+1}, else D_{j+1} zero -> B_j. "Zero" is the masked zero test of the whole frame at thr.
//
// Three parts, a fixed number of launches whatever S and L:
//   1. ofk_nonzero_flags of every input frame (probe + scan).
//   2. acc_walk: a CTA owns a 32 x 32 tile of one clip and walks it through all L steps with the running flow (u, v,
//      mask) in registers: per step every tap gather of the thread's rows is issued before the first use, the state is
//      written coalesced when cumulative, and its zero test is published per (clip, step). The exits the input flags
//      decide are exact here: restart from an input, pass-through of the state, and a state known to be zero because
//      it restarted from a zero input. A composed state is assumed to be non-zero.
//   3. acc_repair: one CTA per clip. A composed state before the last step that is zero on all its valid pixels
//      (cancellation, e.g. a translation followed by its inverse) makes combine_with restart from the next input,
//      which the walk cannot know in advance. The CTA compares the published flags with the walk's assumption and
//      returns at once when none failed (the normal case); otherwise it redoes its clip from that step, one frame pass
//      per step with CTA-wide zero tests, keeping the state in `out` (the clip's frames when cumulative, its one
//      output frame, rebuilt from the first step, otherwise). Slow (one SM per affected clip) but exact.
#include "combine3_device.cuh"

namespace ofk {
namespace acc {

constexpr int kRows = 4;          // rows per thread: 8 warps x 4 rows x 32 lanes = a 32 x 32 tile per CTA
constexpr int kThreads = 256;
constexpr int kRepairThreads = 1024;

struct State {
    float u[kRows], v[kRows];
    unsigned m[kRows];
};

// frame index of walk step `step` (the right fold walks the clip backwards)
template <bool REF_T>
__device__ __forceinline__ int frame_of(int step, int L) { return REF_T ? L - 1 - step : step; }

__device__ __forceinline__ bool nonzero_at(float u, float v, unsigned m, float tz) {
    return m && (fabsf(u) >= tz || fabsf(v) >= tz);
}

// One composition step of the rows of a thread: state += Q(G, p + sign * state), mask &= strict(Gm at the taps). The
// same arithmetic as process_tile (combine3.cu): the interior path when every tap of the warp is inside the frame, the
// exact per-pixel sample otherwise.
template <bool REF_T>
__device__ __forceinline__ void compose(State& s, const float2* __restrict__ G, const uint8_t* __restrict__ Gm,
                                        float Xg, const float* Yg, int H, int W) {
    const float sign = REF_T ? -1.0f : 1.0f;
    float X[kRows], Y[kRows];
    QCoord qx[kRows], qy[kRows];
    bool interior = true;
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
        X[j] = __fmaf_rn(sign, s.u[j], Xg);
        Y[j] = __fmaf_rn(sign, s.v[j], Yg[j]);
        qx[j] = quantise_fast(X[j]);
        qy[j] = quantise_fast(Y[j]);
        interior = interior && (unsigned)qx[j].i < (unsigned)(W - 1) && (unsigned)qy[j].i < (unsigned)(H - 1) &&
                   fabsf(X[j]) < OFK_FAST_COORD_LIMIT && fabsf(Y[j]) < OFK_FAST_COORD_LIMIT;
    }
    float su[kRows], sv[kRows];
    unsigned strict[kRows];
    if (__all_sync(0xffffffffu, interior)) {
        float2 tp[kRows][4];
        unsigned inv[kRows][4];
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            const unsigned o = (unsigned)(qy[j].i * W + qx[j].i);
            const float2* g0 = G + o;
            const float2* g1 = g0 + W;
            tp[j][0] = __ldg(g0); tp[j][1] = __ldg(g0 + 1); tp[j][2] = __ldg(g1); tp[j][3] = __ldg(g1 + 1);
            const uint8_t* m0 = Gm + o;
            const uint8_t* m1 = m0 + W;
            inv[j][0] = __ldg(m0); inv[j][1] = __ldg(m0 + 1); inv[j][2] = __ldg(m1); inv[j][3] = __ldg(m1 + 1);
        }
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            const int a = qx[j].f, b = qy[j].f;
            const unsigned za = a == 0, zb = b == 0;
            strict[j] = inv[j][0] & (inv[j][1] | za) & (inv[j][2] | zb) & (inv[j][3] | za | zb);
            const float fa = (float)a * (1.0f / 32.0f), fb = (float)b * (1.0f / 32.0f);
            const float na = 1.0f - fa, nb = 1.0f - fb;
            const float f00 = __fmul_rn(na, nb), f01 = __fmul_rn(fa, nb), f10 = __fmul_rn(na, fb),
                        f11 = __fmul_rn(fa, fb);
            su[j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(tp[j][0].x, f00), __fmul_rn(tp[j][1].x, f01)),
                                        __fmul_rn(tp[j][2].x, f10)), __fmul_rn(tp[j][3].x, f11));
            sv[j] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(tp[j][0].y, f00), __fmul_rn(tp[j][1].y, f01)),
                                        __fmul_rn(tp[j][2].y, f10)), __fmul_rn(tp[j][3].y, f11));
        }
    } else {
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            const SampleResult r = sample_flow_border(G, Gm, H, W, X[j], Y[j]);
            su[j] = r.u; sv[j] = r.v; strict[j] = (unsigned)r.strict;
        }
    }
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
        s.u[j] = __fadd_rn(s.u[j], su[j]);
        s.v[j] = __fadd_rn(s.v[j], sv[j]);
        s.m[j] &= strict[j];
    }
}

// Grid: S * tiles CTAs (clip-major), dynamic shared memory: one bit per step of the clip.
//   in_nz [S*L]: input zero flags; st_nz [S*L] (zeroed): receives 1 where the state of (clip, step) is non-zero.
// Three CTAs per SM (80 registers, no spills; with four, ptxas caps the walk at 64 registers and spills).
template <bool REF_T, bool CUM>
__global__ void __launch_bounds__(kThreads, 3) acc_walk(const float2* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                        const int* __restrict__ in_nz, float tz, int L, int H, int W,
                                                        int tiles_x, int tiles, float2* __restrict__ out,
                                                        uint8_t* __restrict__ out_mask, int* __restrict__ st_nz) {
    extern __shared__ unsigned nz_bits[];
    const int words = (L + 31) >> 5;
    for (int i = threadIdx.x; i < words; i += kThreads) nz_bits[i] = 0;
    __syncthreads();

    const int s = blockIdx.x / tiles, t = blockIdx.x - s * tiles;
    const int ty = t / tiles_x, tx = t - ty * tiles_x;
    const unsigned lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const unsigned x = (unsigned)tx * 32 + lane, y0 = (unsigned)ty * 32 + wrp * kRows;
    // threads past the frame border walk the border pixel (same frame, so no false non-zero flags) and store nothing
    const unsigned xc = min(x, (unsigned)W - 1);
    const float Xg = static_cast<float>(xc);
    float Yg[kRows];
    unsigned idx[kRows];
#pragma unroll
    for (int j = 0; j < kRows; ++j) {
        const unsigned yc = min(y0 + j, (unsigned)H - 1);
        Yg[j] = static_cast<float>(yc);
        idx[j] = yc * (unsigned)W + xc;
    }
    const size_t frame = (size_t)H * W;
    const size_t clip0 = (size_t)s * L;
    const int* nzB = in_nz + clip0;

    State st;
    bool zero = false;   // the state is known to be zero (a restart from a zero input)
    for (int step = 0; step < L; ++step) {
        const int k = frame_of<REF_T>(step, L);
        const bool nzb = nzB[k] != 0;
        const float2* G = B + (clip0 + k) * frame;
        const uint8_t* Gm = Bm + (clip0 + k) * frame;
        // REF_T: B_k zero -> pass, else state zero -> restart; otherwise: state zero -> restart, else B_k zero -> pass
        const bool restart = step == 0 || (REF_T ? (nzb && zero) : zero);
        const bool pass = !restart && !nzb;
        if (restart) {
#pragma unroll
            for (int j = 0; j < kRows; ++j) {
                const float2 f = ld_stream_f2(G + idx[j]);
                st.u[j] = f.x;
                st.v[j] = f.y;
                st.m[j] = Gm[idx[j]];
            }
            zero = !nzb;
        } else if (!pass) {
            compose<REF_T>(st, G, Gm, Xg, Yg, H, W);
        }
        bool nz = false;
#pragma unroll
        for (int j = 0; j < kRows; ++j) nz |= nonzero_at(st.u[j], st.v[j], st.m[j], tz);
        if (__any_sync(0xffffffffu, nz) && lane == 0) atomicOr(&nz_bits[k >> 5], 1u << (k & 31));
        if (CUM && x < (unsigned)W) {
            float2* O = out + (clip0 + k) * frame;
            uint8_t* Om = out_mask + (clip0 + k) * frame;
#pragma unroll
            for (int j = 0; j < kRows; ++j) {
                if (y0 + j < (unsigned)H) {
                    asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(O + idx[j]), "f"(st.u[j]),
                                 "f"(st.v[j])
                                 : "memory");
                    Om[idx[j]] = (uint8_t)st.m[j];
                }
            }
        }
    }
    if (!CUM && x < (unsigned)W) {
        float2* O = out + (size_t)s * frame;
        uint8_t* Om = out_mask + (size_t)s * frame;
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            if (y0 + j < (unsigned)H) {
                O[idx[j]] = make_float2(st.u[j], st.v[j]);
                Om[idx[j]] = (uint8_t)st.m[j];
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < words; i += kThreads) {
        unsigned bits = nz_bits[i];
        while (bits) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            st_nz[clip0 + i * 32 + b] = 1;   // benign race: every writer stores the same value
        }
    }
}

// The exact fold of one clip from walk step `first`, one frame pass per step. The state of the previous step is in
// frame `prev` of out (in place when not cumulative); `zero` is its exact zero test.
template <bool REF_T, bool CUM>
__device__ void redo_clip(const float2* __restrict__ B, const uint8_t* __restrict__ Bm, const int* __restrict__ nzB,
                          float tz, int L, int H, int W, int first, bool zero, float2* out, uint8_t* out_mask,
                          size_t clip0, size_t out_clip0) {
    const unsigned frame = (unsigned)H * (unsigned)W;
    for (int step = first; step < L; ++step) {
        const int k = frame_of<REF_T>(step, L);
        const bool nzb = nzB[k] != 0;
        const float2* G = B + (clip0 + k) * frame;
        const uint8_t* Gm = Bm + (clip0 + k) * frame;
        float2* P = out + (out_clip0 + (CUM ? frame_of<REF_T>(step - 1, L) : 0)) * frame;   // step 0: unused
        uint8_t* Pm = out_mask + (out_clip0 + (CUM ? frame_of<REF_T>(step - 1, L) : 0)) * frame;
        float2* O = out + (out_clip0 + (CUM ? k : 0)) * frame;
        uint8_t* Om = out_mask + (out_clip0 + (CUM ? k : 0)) * frame;
        const bool restart = step == 0 || (REF_T ? (nzb && zero) : zero);
        const bool pass = !restart && !nzb;
        if (restart || pass) {
            if (restart || CUM) {
                const float2* src = restart ? G : P;
                const uint8_t* srcm = restart ? Gm : Pm;
                for (unsigned i = threadIdx.x; i < frame; i += kRepairThreads) {
                    O[i] = src[i];
                    Om[i] = srcm[i];
                }
            }
            if (restart) zero = !nzb;
            continue;
        }
        bool nz = false;
        for (unsigned i = threadIdx.x; i < frame; i += kRepairThreads) {
            const unsigned y = i / (unsigned)W, x = i - y * (unsigned)W;
            const float2 p = P[i];
            const float sign = REF_T ? -1.0f : 1.0f;
            const SampleResult r = sample_flow_border(G, Gm, H, W, __fmaf_rn(sign, p.x, (float)x),
                                                      __fmaf_rn(sign, p.y, (float)y));
            const float u = __fadd_rn(p.x, r.u), v = __fadd_rn(p.y, r.v);
            const unsigned m = Pm[i] & (unsigned)r.strict;
            O[i] = make_float2(u, v);
            Om[i] = (uint8_t)m;
            nz |= nonzero_at(u, v, m, tz);
        }
        zero = !__syncthreads_or(nz);
    }
}

template <bool REF_T, bool CUM>
__global__ void __launch_bounds__(kRepairThreads) acc_repair(const float2* __restrict__ B,
                                                             const uint8_t* __restrict__ Bm,
                                                             const int* __restrict__ in_nz,
                                                             const int* __restrict__ st_nz, float tz, int L, int H,
                                                             int W, float2* out, uint8_t* out_mask) {
    const int s = blockIdx.x;
    const size_t clip0 = (size_t)s * L;
    const int* nzB = in_nz + clip0;
    const int* nzS = st_nz + clip0;
    // replay the walk's decisions: the first step before the last whose composed state was assumed non-zero but is not
    bool zero = nzB[frame_of<REF_T>(0, L)] == 0;
    int failed = -1;
    for (int step = 1; step < L - 1; ++step) {
        const int k = frame_of<REF_T>(step, L);
        const bool nzb = nzB[k] != 0;
        const bool restart = REF_T ? (nzb && zero) : zero;
        if (restart) {
            zero = !nzb;
        } else if (nzb && nzS[k] == 0) {
            failed = step;
            break;
        }
    }
    if (failed < 0) return;
    if (CUM) redo_clip<REF_T, true>(B, Bm, nzB, tz, L, H, W, failed + 1, true, out, out_mask, clip0, clip0);
    else redo_clip<REF_T, false>(B, Bm, nzB, tz, L, H, W, 0, false, out, out_mask, clip0, (size_t)s);
}

struct Layout {
    size_t in_nz, st_nz, total;
};
static Layout layout(int S, int L) {
    const size_t flags = ((size_t)S * L * sizeof(int) + 255) & ~(size_t)255;
    return Layout{0, flags, 2 * flags};
}

}  // namespace acc
}  // namespace ofk

using namespace ofk;

extern "C" size_t ofk_accumulate_workspace(int S, int L) {
    if (S < 0 || L < 1 || (long long)S * L > 65535) return 0;
    return acc::layout(S, L).total;
}

extern "C" int ofk_accumulate(const float* flow, const uint8_t* mask, int ref, float thr, int S, int L, int H, int W,
                              int cumulative, float* out, uint8_t* out_mask, void* ws, size_t ws_bytes,
                              ofk_stream_t stream) {
    OFK_CHECK_ARG(flow && mask && out && out_mask && ws, "ofk_accumulate: NULL pointer");
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofk_accumulate: ref must be 's' or 't', got %d", ref);
    OFK_CHECK_ARG(thr >= 0.f, "ofk_accumulate: thr must be >= 0");
    OFK_CHECK_ARG(S >= 0 && L >= 1 && H > 0 && W > 0 && H < 32768 && W < 32768,
                  "ofk_accumulate: bad shape S=%d L=%d H=%d W=%d (L >= 1, H and W below 32768)", S, L, H, W);
    OFK_CHECK_ARG((long long)S * L <= 65535, "ofk_accumulate: S*L = %lld exceeds 65535 frames per call",
                  (long long)S * L);
    const long long tiles = (long long)((W + 31) / 32) * ((H + 31) / 32);
    OFK_CHECK_ARG((long long)S * tiles <= 0x7fffffffLL, "ofk_accumulate: too many tiles (S=%d H=%d W=%d)", S, H, W);
    OFK_CHECK_ARG(((reinterpret_cast<uintptr_t>(flow) | reinterpret_cast<uintptr_t>(out)) & 7) == 0,
                  "ofk_accumulate: flow and out must be 8-byte aligned");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 3) == 0, "ofk_accumulate: ws must be 4-byte aligned");
    const acc::Layout lay = acc::layout(S, L);
    OFK_CHECK_ARG(ws_bytes >= lay.total, "ofk_accumulate: workspace too small (%zu bytes, need %zu)", ws_bytes,
                  lay.total);
    if (S == 0) return OFK_OK;
    cudaStream_t st = as_stream(stream);
    const int N = S * L;
    int* in_nz = reinterpret_cast<int*>(static_cast<char*>(ws) + lay.in_nz);
    int* st_nz = reinterpret_cast<int*>(static_cast<char*>(ws) + lay.st_nz);
    const int rc = ofk_nonzero_flags(flow, mask, thr, in_nz, N, H, W, stream);
    if (rc != OFK_OK) return rc;
    OFK_CUDA(cudaMemsetAsync(st_nz, 0, sizeof(int) * (size_t)N, st));
    // zero test as one compare per component: |c| >= t with t = thr, or the smallest denormal for the exact test
    const float tz = thr > 0.f ? thr : 1.401298464e-45f;
    const float2* B = reinterpret_cast<const float2*>(flow);
    float2* O = reinterpret_cast<float2*>(out);
    const int tiles_x = (W + 31) / 32;
    const unsigned grid = (unsigned)(S * tiles);
    const size_t smem = sizeof(unsigned) * (size_t)((L + 31) / 32);
#define OFK_ACC(RT, CU)                                                                                              \
    do {                                                                                                             \
        acc::acc_walk<RT, CU><<<grid, acc::kThreads, smem, st>>>(B, mask, in_nz, tz, L, H, W, tiles_x, (int)tiles,  \
                                                                 O, out_mask, st_nz);                                \
        OFK_LAUNCHED();                                                                                              \
        acc::acc_repair<RT, CU><<<S, acc::kRepairThreads, 0, st>>>(B, mask, in_nz, st_nz, tz, L, H, W, O, out_mask); \
        OFK_LAUNCHED();                                                                                              \
    } while (0)
    if (ref == 't') {
        if (cumulative) OFK_ACC(true, true);
        else OFK_ACC(true, false);
    } else {
        if (cumulative) OFK_ACC(false, true);
        else OFK_ACC(false, false);
    }
#undef OFK_ACC
    return OFK_OK;
}
