// Flow error metrics of N estimates against their ground truth, ofk_evaluate: end-point error, angular error, the
// KITTI Fl and 1 / 3 / 5 px outlier counts and the Sintel speed bands, per frame, in two launches whatever N.
//
//   eval_kernel   : one CTA per fixed block of kBlockPx pixels of one frame (grid x: block, grid y: frame). Every
//                   thread takes groups of 4 consecutive pixels, accumulates its counts in int32 and its sums in
//                   float64 in pixel order, and the CTA reduces them in a fixed order (warp tree, then warps 0..7) to
//                   one Partial. The per-pixel arithmetic is float32 with explicit _rn intrinsics, so that nothing is
//                   contracted into an FMA and a numpy float32 restatement reproduces it bit for bit.
//   finish_kernel : one warp per frame sums the frame's partials in block order (counts widened to int64).
// A group is loaded with 16-byte vector loads where the frame's first pixel is 4-aligned in every array (and the bases
// allow), else with scalar loads; both paths visit the same pixels in the same order per thread, so a frame's rows do
// not depend on its position in the batch.
#include <math.h>

#include "ofk_common.cuh"

namespace ofk {
namespace {

constexpr int kThreads = 256;
constexpr int kBlockPx = 8192;                          // fixed: the partials of a frame do not depend on the batch
constexpr int kGroups = kBlockPx / (4 * kThreads);      // groups of 4 pixels per thread and block
constexpr int kFramesPerFinish = 4;                     // warps (frames) per block of finish_kernel

struct Partial {        // one block: sums {epe, ae, epe band 0, 1, 2}, counts {n, fl, >1, >3, >5, band 0, 1, 2}
    double s[5];
    int c[8];
};

struct Acc {
    double epe = 0.0, ae = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0;
    int n = 0, fl = 0, o1 = 0, o3 = 0, o5 = 0, c0 = 0, c1 = 0, c2 = 0;
};

// The metrics of one pixel (the definitions of include/oflib_b200.h); returns its EPE, accumulates it where ev.
__device__ __forceinline__ float pixel(float ue, float ve, float ug, float vg, bool ev, Acc& a) {
    const float du = __fsub_rn(ue, ug), dv = __fsub_rn(ve, vg);
    const float d2 = __fadd_rn(__fmul_rn(du, du), __fmul_rn(dv, dv));
    const float epe = __fsqrt_rn(d2);
    if (ev) {
        const float mg = __fsqrt_rn(__fadd_rn(__fmul_rn(ug, ug), __fmul_rn(vg, vg)));
        const float cz = __fsub_rn(__fmul_rn(ue, vg), __fmul_rn(ve, ug));
        const float cr = __fsqrt_rn(__fadd_rn(d2, __fmul_rn(cz, cz)));
        const float dot = __fadd_rn(__fadd_rn(1.0f, __fmul_rn(ue, ug)), __fmul_rn(ve, vg));
        const float ae = __fmul_rn(atan2f(cr, dot), 57.29578f);
        const double e = (double)epe;
        a.n += 1;
        a.epe += e;
        a.ae += (double)ae;
        a.o1 += epe > 1.0f;
        a.o3 += epe > 3.0f;
        a.o5 += epe > 5.0f;
        if (epe > 3.0f && __fdiv_rn(epe, mg) > 0.05f) a.fl += 1;    // mg = 0: epe / 0 = inf
        const bool lo = mg < 10.0f, mid = !lo && mg < 40.0f, hi = !(mg < 40.0f);
        a.c0 += lo;
        a.c1 += mid;
        a.c2 += hi;
        a.b0 += lo ? e : 0.0;
        a.b1 += mid ? e : 0.0;
        a.b2 += hi ? e : 0.0;
    }
    return epe;
}

template <bool EM, bool TM, bool RG, bool MAP>
__global__ void __launch_bounds__(kThreads) eval_kernel(const float* __restrict__ est, const uint8_t* __restrict__ em,
                                                        const float* __restrict__ truth,
                                                        const uint8_t* __restrict__ tm,
                                                        const uint8_t* __restrict__ rg, float* __restrict__ epe,
                                                        Partial* __restrict__ part, int hw, int vec_base) {
    const size_t fbase = (size_t)blockIdx.y * hw;
    const int p0 = blockIdx.x * kBlockPx;
    const bool vec = vec_base && (fbase & 3) == 0;
    Acc a;
#pragma unroll 2
    for (int k = 0; k < kGroups; ++k) {
        const int q = p0 + (k * kThreads + threadIdx.x) * 4;      // first pixel of the group, in the frame
        if (q >= hw) break;
        const size_t g = fbase + q;
        if (vec && q + 4 <= hw) {
            const float4 e0 = ld_stream_f4(reinterpret_cast<const float4*>(est + 2 * g));
            const float4 e1 = ld_stream_f4(reinterpret_cast<const float4*>(est + 2 * g) + 1);
            const float4 t0 = ld_stream_f4(reinterpret_cast<const float4*>(truth + 2 * g));
            const float4 t1 = ld_stream_f4(reinterpret_cast<const float4*>(truth + 2 * g) + 1);
            uint32_t m = 0x01010101u;
            if (EM) m &= ld_stream_u32(reinterpret_cast<const uint32_t*>(em + g));
            if (TM) m &= ld_stream_u32(reinterpret_cast<const uint32_t*>(tm + g));
            if (RG) m &= ld_stream_u32(reinterpret_cast<const uint32_t*>(rg + g));
            float4 r;
            r.x = pixel(e0.x, e0.y, t0.x, t0.y, (m & 0xffu) != 0, a);
            r.y = pixel(e0.z, e0.w, t0.z, t0.w, (m & 0xff00u) != 0, a);
            r.z = pixel(e1.x, e1.y, t1.x, t1.y, (m & 0xff0000u) != 0, a);
            r.w = pixel(e1.z, e1.w, t1.z, t1.w, (m & 0xff000000u) != 0, a);
            if (MAP) st_stream_f4(reinterpret_cast<float4*>(epe + g), r);
        } else {
            const int cnt = min(4, hw - q);
            for (int j = 0; j < cnt; ++j) {
                const float2 e = reinterpret_cast<const float2*>(est)[g + j];
                const float2 t = reinterpret_cast<const float2*>(truth)[g + j];
                bool ev = true;
                if (EM) ev = ev && em[g + j] != 0;
                if (TM) ev = ev && tm[g + j] != 0;
                if (RG) ev = ev && rg[g + j] != 0;
                const float r = pixel(e.x, e.y, t.x, t.y, ev, a);
                if (MAP) epe[g + j] = r;
            }
        }
    }
    // fixed-order reduction: a shuffle tree per warp, then the warps in order
    __shared__ double ws[kThreads / 32][5];
    __shared__ int wc[kThreads / 32][8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double s[5] = {a.epe, a.ae, a.b0, a.b1, a.b2};
    const int c[8] = {a.n, a.fl, a.o1, a.o3, a.o5, a.c0, a.c1, a.c2};
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        for (int o = 16; o > 0; o >>= 1) s[i] += __shfl_down_sync(0xffffffffu, s[i], o);
        if (lane == 0) ws[wid][i] = s[i];
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int t = __reduce_add_sync(0xffffffffu, c[i]);
        if (lane == 0) wc[wid][i] = t;
    }
    __syncthreads();
    Partial& out = part[(size_t)blockIdx.y * gridDim.x + blockIdx.x];
    if (threadIdx.x < 5) {
        double t = ws[0][threadIdx.x];
        for (int w = 1; w < kThreads / 32; ++w) t += ws[w][threadIdx.x];
        out.s[threadIdx.x] = t;
    } else if (threadIdx.x >= 32 && threadIdx.x < 40) {
        const int i = threadIdx.x - 32;
        int t = 0;
        for (int w = 0; w < kThreads / 32; ++w) t += wc[w][i];
        out.c[i] = t;
    }
}

// One warp per frame: lane i < 8 sums count i, lanes 8..12 sum i - 8, over the frame's blocks in order.
__global__ void __launch_bounds__(32 * kFramesPerFinish) finish_kernel(const Partial* __restrict__ part,
                                                                      long long* __restrict__ counts,
                                                                      double* __restrict__ sums, int N, int bpf) {
    const int n = blockIdx.x * kFramesPerFinish + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N || lane >= 13) return;
    const Partial* p = part + (size_t)n * bpf;
    if (lane < 8) {
        long long t = 0;
        for (int b = 0; b < bpf; ++b) t += p[b].c[lane];
        counts[(size_t)n * 8 + lane] = t;
    } else {
        double t = 0.0;
        for (int b = 0; b < bpf; ++b) t += p[b].s[lane - 8];
        sums[(size_t)n * 5 + lane - 8] = t;
    }
}

template <bool EM, bool TM, bool RG, bool MAP>
void launch(dim3 grid, cudaStream_t st, const float* est, const uint8_t* em, const float* truth, const uint8_t* tm,
            const uint8_t* rg, float* epe, Partial* part, int hw, int vec_base) {
    eval_kernel<EM, TM, RG, MAP><<<grid, kThreads, 0, st>>>(est, em, truth, tm, rg, epe, part, hw, vec_base);
}

using LaunchFn = void (*)(dim3, cudaStream_t, const float*, const uint8_t*, const float*, const uint8_t*,
                          const uint8_t*, float*, Partial*, int, int);

template <int I>
constexpr LaunchFn variant() {
    return &launch<(I & 1) != 0, (I & 2) != 0, (I & 4) != 0, (I & 8) != 0>;
}
constexpr LaunchFn kVariants[16] = {variant<0>(),  variant<1>(),  variant<2>(),  variant<3>(),
                                    variant<4>(),  variant<5>(),  variant<6>(),  variant<7>(),
                                    variant<8>(),  variant<9>(),  variant<10>(), variant<11>(),
                                    variant<12>(), variant<13>(), variant<14>(), variant<15>()};

bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }
bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

size_t blocks_per_frame(int H, int W) { return ((size_t)H * W + kBlockPx - 1) / kBlockPx; }

}  // namespace
}  // namespace ofk

using namespace ofk;

extern "C" size_t ofk_evaluate_workspace(int N, int H, int W) {
    if (N < 0 || N > 65535 || H <= 0 || W <= 0 || (size_t)H * W >= (1ull << 31)) return 0;
    return (size_t)N * blocks_per_frame(H, W) * sizeof(Partial);
}

extern "C" int ofk_evaluate(const float* est, const uint8_t* est_mask, const float* truth, const uint8_t* truth_mask,
                            const uint8_t* region, float* epe, long long* counts, double* sums, int N, int H, int W,
                            void* ws, size_t ws_bytes, ofk_stream_t stream) {
    OFK_CHECK_ARG(est && truth && counts && sums,
                  "ofk_evaluate: NULL pointer (est, truth, counts and sums are required)");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0, "ofk_evaluate: bad shape");
    OFK_CHECK_ARG(N <= 65535, "ofk_evaluate: N = %d exceeds 65535 frames", N);
    OFK_CHECK_ARG((size_t)H * W < (1ull << 31), "ofk_evaluate: a frame needs fewer than 2^31 pixels");
    OFK_CHECK_ARG(aligned8(est) && aligned8(truth), "ofk_evaluate: est and truth must be 8-byte aligned");
    OFK_CHECK_ARG(aligned8(counts) && aligned8(sums), "ofk_evaluate: counts and sums must be 8-byte aligned");
    OFK_CHECK_ARG(epe == nullptr || aligned4(epe), "ofk_evaluate: epe must be 4-byte aligned");
    const size_t need = ofk_evaluate_workspace(N, H, W);
    OFK_CHECK_ARG(N == 0 || (ws != nullptr && aligned8(ws) && ws_bytes >= need),
                  "ofk_evaluate: workspace needs %zu bytes, 8-byte aligned (got %zu)", need, ws_bytes);
    if (N == 0) return OFK_OK;
    const int hw = H * W;
    const int bpf = (int)blocks_per_frame(H, W);
    const int vec_base = aligned16(est) && aligned16(truth) && (!est_mask || aligned4(est_mask)) &&
                         (!truth_mask || aligned4(truth_mask)) && (!region || aligned4(region)) &&
                         (!epe || aligned16(epe));
    const int v = (est_mask ? 1 : 0) | (truth_mask ? 2 : 0) | (region ? 4 : 0) | (epe ? 8 : 0);
    Partial* part = static_cast<Partial*>(ws);
    const cudaStream_t st = as_stream(stream);
    kVariants[v](dim3(bpf, N), st, est, est_mask, truth, truth_mask, region, epe, part, hw, vec_base);
    OFK_LAUNCHED();
    finish_kernel<<<(N + kFramesPerFinish - 1) / kFramesPerFinish, 32 * kFramesPerFinish, 0, st>>>(part, counts, sums,
                                                                                                 N, bpf);
    OFK_LAUNCHED();
    return OFK_OK;
}
