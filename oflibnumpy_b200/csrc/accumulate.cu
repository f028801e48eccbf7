// Accumulation of clips of flows to their keyframe, mode-3 composition folded over each clip (ofk_accumulate,
// ofk_accumulate_fold).
//
// A batch of S*L frames is S clips of L consecutive frames B_0 .. B_{L-1}. Mode 3 reads one operand at p and samples
// the other (combine3.cu). Two of the four (ref, fold) combinations read the running flow at p, so they are pointwise
// in it and can be walked:
//   ref 's' (left fold):  C_0 = B_0,      C_k = C_{k-1} (+) B_k:  C_k(p) = C_{k-1}(p) + Q(B_k, p + C_{k-1}(p))
//   ref 't' (right fold): D_{L-1} = B_{L-1}, D_j = B_j (+) D_{j+1}: D_j(p) = D_{j+1}(p) + Q(B_j, p - D_{j+1}(p))
// The other two sample the running flow, so every step needs the previous composite of the whole frame:
//   ref 't' (left fold):  E_0 = B_0,      E_k = E_{k-1} (+) B_k:  E_k(p) = B_k(p) + Q(E_{k-1}, p - B_k(p))
//   ref 's' (right fold): R_{L-1} = B_{L-1}, R_j = B_j (+) R_{j+1}: R_j(p) = B_j(p) + Q(R_{j+1}, p + B_j(p))
// with the early exits of combine_with (self tested first), which depend on the fold only: left fold, state zero ->
// B_k, else B_k zero -> state; right fold, B_j zero -> state, else state zero -> B_j. "Zero" is the masked zero test of
// the whole frame at thr.
//
// Walked combinations, a fixed number of launches whatever S and L:
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
// Sampled combinations, one launch per step:
//   1. ofk_nonzero_flags of every input frame, as above.
//   2. acc_step, once per step for all S clips: a CTA owns a 32 x 32 tile of one clip, loads B_k as the state and
//      composes it with the previous step's frame. The previous step's zero flag, final by stream order, decides
//      restart, pass or compose for the whole clip before anything else is read; a composing step publishes its own.
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

// Frame k of clip s of a frame array: v + (s * clip_stride + k) * H*W (clip_stride L for a batch, 1 for one frame
// per clip).
struct Src {
    const float2* v;
    const uint8_t* m;
    size_t clip_stride;
    int k;
};
struct Dst {
    float2* v;
    uint8_t* m;
    size_t clip_stride;
    int k;
};

// One step of a sampled combination for all S clips. Grid: S * tiles CTAs (clip-major).
//   REF_T (ref 't', left fold):  k = step,     exits: state zero -> restart, else B_k zero -> pass.
//   !REF_T (ref 's', right fold): k = L-1-step, exits: B_k zero -> pass, else state zero -> restart.
// `first` forces the restart (the clip's anchor frame). P is the previous step's frame, of frame index kp, and
// p_nz[s*L + kp] its zero flag. The result goes to frame O.k of O and its flag to st_nz[s*L + k] (zeroed by the call):
// a copying step writes the flag whole, a composing step sets it where a CTA sees a non-zero pixel.
// Four CTAs per SM (64 registers, no spills): with no state carried between steps it fits where the walk does not.
template <bool REF_T>
__global__ void __launch_bounds__(kThreads, 4) acc_step(const float2* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                        const int* __restrict__ in_nz, int k, bool first, Src P,
                                                        const int* p_nz, int kp, Dst O, int* st_nz, float tz, int L,
                                                        int H, int W, int tiles_x, int tiles) {
    const int s = blockIdx.x / tiles, t = blockIdx.x - s * tiles;
    const int ty = t / tiles_x, tx = t - ty * tiles_x;
    const unsigned lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const unsigned x = (unsigned)tx * 32 + lane, y0 = (unsigned)ty * 32 + wrp * kRows;
    // threads past the frame border compose the border pixel (same frame, so no false non-zero flags), store nothing
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
    const bool nzb = in_nz[clip0 + k] != 0;
    const bool zero = !first && p_nz[clip0 + kp] == 0;
    const bool restart = first || (REF_T ? zero : (nzb && zero));
    const bool pass = !restart && !nzb;
    const float2* G = B + (clip0 + k) * frame;
    const uint8_t* Gm = Bm + (clip0 + k) * frame;
    const float2* Pv = P.v + ((size_t)s * P.clip_stride + P.k) * frame;
    const uint8_t* Pm = P.m + ((size_t)s * P.clip_stride + P.k) * frame;
    float2* Ov = O.v + ((size_t)s * O.clip_stride + O.k) * frame;
    uint8_t* Om = O.m + ((size_t)s * O.clip_stride + O.k) * frame;

    State st;
    if (restart || pass) {
        if (t == 0 && threadIdx.x == 0) st_nz[clip0 + k] = restart ? nzb : !zero;
        const float2* src = restart ? G : Pv;
        const uint8_t* srcm = restart ? Gm : Pm;
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            const float2 f = ld_stream_f2(src + idx[j]);
            st.u[j] = f.x;
            st.v[j] = f.y;
            st.m[j] = srcm[idx[j]];
        }
    } else {
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            const float2 f = ld_stream_f2(G + idx[j]);
            st.u[j] = f.x;
            st.v[j] = f.y;
            st.m[j] = Gm[idx[j]];
        }
        compose<REF_T>(st, Pv, Pm, Xg, Yg, H, W);
    }
    if (x < (unsigned)W) {
#pragma unroll
        for (int j = 0; j < kRows; ++j) {
            if (y0 + j < (unsigned)H) {
                asm volatile("st.global.L1::no_allocate.v2.f32 [%0], {%1,%2};" ::"l"(Ov + idx[j]), "f"(st.u[j]),
                             "f"(st.v[j])
                             : "memory");
                Om[idx[j]] = (uint8_t)st.m[j];
            }
        }
    }
    if (restart || pass) return;
    bool nz = false;
#pragma unroll
    for (int j = 0; j < kRows; ++j) nz |= nonzero_at(st.u[j], st.v[j], st.m[j], tz);
    // Every CTA of the clip publishes to the same int. Same-address stores serialise in L2, so store once per CTA,
    // and only while the flag is not yet set (benign race: every writer stores 1).
    if (__syncthreads_or(nz) && threadIdx.x == 0 && __ldcg(st_nz + clip0 + k) == 0) st_nz[clip0 + k] = 1;
}

struct Layout {
    size_t in_nz, st_nz, buf, buf_mask, total;
};
// Two int flag arrays of S*L; the sampled combinations, when not cumulative, add one S-frame buffer that alternates
// with out between the steps.
static Layout layout(int S, int L, bool buffer = false, int H = 0, int W = 0) {
    const auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t flags = up((size_t)S * L * sizeof(int));
    const size_t px = buffer ? (size_t)S * H * W : 0;
    const size_t buf_mask = 2 * flags + up(px * sizeof(float2));
    return Layout{0, flags, 2 * flags, buf_mask, buf_mask + up(px)};
}

// The sampled combinations: ref 't' with the left fold, ref 's' with the right fold.
static bool sampled(int ref, int fold) { return (ref == 't') == (fold == 'l'); }

static int check_args(const char* fn, const float* flow, const uint8_t* mask, int ref, int fold, float thr, int S,
                      int L, int H, int W, int cumulative, const float* out, const uint8_t* out_mask, const void* ws,
                      size_t ws_bytes) {
    OFK_CHECK_ARG(flow && mask && out && out_mask && ws, "%s: NULL pointer", fn);
    OFK_CHECK_ARG(ref == 's' || ref == 't', "%s: ref must be 's' or 't', got %d", fn, ref);
    OFK_CHECK_ARG(fold == 'l' || fold == 'r', "%s: fold must be 'l' or 'r', got %d", fn, fold);
    OFK_CHECK_ARG(thr >= 0.f, "%s: thr must be >= 0", fn);
    OFK_CHECK_ARG(S >= 0 && L >= 1 && H > 0 && W > 0 && H < 32768 && W < 32768,
                  "%s: bad shape S=%d L=%d H=%d W=%d (L >= 1, H and W below 32768)", fn, S, L, H, W);
    OFK_CHECK_ARG((long long)S * L <= 65535, "%s: S*L = %lld exceeds 65535 frames per call", fn, (long long)S * L);
    const long long tiles = (long long)((W + 31) / 32) * ((H + 31) / 32);
    OFK_CHECK_ARG((long long)S * tiles <= 0x7fffffffLL, "%s: too many tiles (S=%d H=%d W=%d)", fn, S, H, W);
    OFK_CHECK_ARG(((reinterpret_cast<uintptr_t>(flow) | reinterpret_cast<uintptr_t>(out)) & 7) == 0,
                  "%s: flow and out must be 8-byte aligned", fn);
    // the sampled combinations keep a float2 frame buffer in the workspace
    const unsigned align = sampled(ref, fold) ? 8 : 4;
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & (align - 1)) == 0, "%s: ws must be %u-byte aligned", fn, align);
    const size_t need = layout(S, L, sampled(ref, fold) && !cumulative, H, W).total;
    OFK_CHECK_ARG(ws_bytes >= need, "%s: workspace too small (%zu bytes, need %zu)", fn, ws_bytes, need);
    return OFK_OK;
}

}  // namespace acc
}  // namespace ofk

using namespace ofk;

// Both folds for checked arguments.
static int accumulate(const float* flow, const uint8_t* mask, int ref, int fold, float thr, int S, int L, int H, int W,
                      int cumulative, float* out, uint8_t* out_mask, void* ws, ofk_stream_t stream) {
    if (S == 0) return OFK_OK;
    const bool sampled = acc::sampled(ref, fold);
    const acc::Layout lay = acc::layout(S, L, sampled && !cumulative, H, W);
    cudaStream_t st = as_stream(stream);
    const int N = S * L;
    char* wsb = static_cast<char*>(ws);
    int* in_nz = reinterpret_cast<int*>(wsb + lay.in_nz);
    int* st_nz = reinterpret_cast<int*>(wsb + lay.st_nz);
    const int rc = ofk_nonzero_flags(flow, mask, thr, in_nz, N, H, W, stream);
    if (rc != OFK_OK) return rc;
    OFK_CUDA(cudaMemsetAsync(st_nz, 0, sizeof(int) * (size_t)N, st));
    // zero test as one compare per component: |c| >= t with t = thr, or the smallest denormal for the exact test
    const float tz = thr > 0.f ? thr : 1.401298464e-45f;
    const float2* B = reinterpret_cast<const float2*>(flow);
    float2* O = reinterpret_cast<float2*>(out);
    const int tiles_x = (W + 31) / 32;
    const int tiles = tiles_x * ((H + 31) / 32);
    const unsigned grid = (unsigned)((long long)S * tiles);
    if (sampled) {
        // Invariant: step i reads the frame step i-1 wrote, and its flag in st_nz, except step 1 of final-only, which
        // reads the anchor input and its flag in in_nz (final-only runs no step 0). Cumulative: step i writes frame k
        // of out. Final-only: the steps alternate between out and the workspace buffer so that the last writes out,
        // and no step writes the buffer it reads.
        const bool left = ref == 't';
        const auto frame_of_step = [&](int i) { return left ? i : L - 1 - i; };
        const auto target = [&](int i) {
            if (cumulative) return acc::Dst{O, out_mask, (size_t)L, frame_of_step(i)};
            if ((L - 1 - i) % 2 == 0) return acc::Dst{O, out_mask, 1, 0};
            return acc::Dst{reinterpret_cast<float2*>(wsb + lay.buf), reinterpret_cast<uint8_t*>(wsb + lay.buf_mask),
                            1, 0};
        };
        for (int i = cumulative || L == 1 ? 0 : 1; i < L; ++i) {
            const int kp = frame_of_step(i == 0 ? 0 : i - 1);                    // step 0 reads no previous frame
            acc::Src P{B, mask, (size_t)L, kp};
            if (i > 1 || (i == 1 && cumulative)) {
                const acc::Dst d = target(i - 1);
                P = acc::Src{d.v, d.m, d.clip_stride, d.k};
            }
            const int* p_nz = i == 1 ? in_nz : st_nz;
            if (left)
                acc::acc_step<true><<<grid, acc::kThreads, 0, st>>>(B, mask, in_nz, frame_of_step(i), i == 0, P, p_nz,
                                                                    kp, target(i), st_nz, tz, L, H, W, tiles_x, tiles);
            else
                acc::acc_step<false><<<grid, acc::kThreads, 0, st>>>(B, mask, in_nz, frame_of_step(i), i == 0, P, p_nz,
                                                                     kp, target(i), st_nz, tz, L, H, W, tiles_x, tiles);
            OFK_LAUNCHED();
        }
        return OFK_OK;
    }
    const size_t smem = sizeof(unsigned) * (size_t)((L + 31) / 32);
#define OFK_ACC(RT, CU)                                                                                              \
    do {                                                                                                             \
        acc::acc_walk<RT, CU><<<grid, acc::kThreads, smem, st>>>(B, mask, in_nz, tz, L, H, W, tiles_x, tiles, O,     \
                                                                 out_mask, st_nz);                                   \
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

extern "C" size_t ofk_accumulate_workspace(int S, int L) {
    if (S < 0 || L < 1 || (long long)S * L > 65535) return 0;
    return acc::layout(S, L).total;
}

extern "C" int ofk_accumulate(const float* flow, const uint8_t* mask, int ref, float thr, int S, int L, int H, int W,
                              int cumulative, float* out, uint8_t* out_mask, void* ws, size_t ws_bytes,
                              ofk_stream_t stream) {
    const int fold = ref == 't' ? 'r' : 'l';
    const int rc = acc::check_args("ofk_accumulate", flow, mask, ref, fold, thr, S, L, H, W, cumulative, out, out_mask,
                                   ws, ws_bytes);
    if (rc != OFK_OK) return rc;
    return accumulate(flow, mask, ref, fold, thr, S, L, H, W, cumulative, out, out_mask, ws, stream);
}

extern "C" size_t ofk_accumulate_fold_workspace(int ref, int fold, int S, int L, int H, int W, int cumulative) {
    if ((ref != 's' && ref != 't') || (fold != 'l' && fold != 'r') || S < 0 || L < 1 || (long long)S * L > 65535 ||
        H <= 0 || W <= 0 || H >= 32768 || W >= 32768)
        return 0;
    return acc::layout(S, L, acc::sampled(ref, fold) && !cumulative, H, W).total;
}

extern "C" int ofk_accumulate_fold(const float* flow, const uint8_t* mask, int ref, int fold, float thr, int S, int L,
                                   int H, int W, int cumulative, float* out, uint8_t* out_mask, void* ws,
                                   size_t ws_bytes, ofk_stream_t stream) {
    const int rc = acc::check_args("ofk_accumulate_fold", flow, mask, ref, fold, thr, S, L, H, W, cumulative, out,
                                   out_mask, ws, ws_bytes);
    if (rc != OFK_OK) return rc;
    return accumulate(flow, mask, ref, fold, thr, S, L, H, W, cumulative, out, out_mask, ws, stream);
}
