// Flow visualisation on the device (SURVEY 8f rank 4): Flow.visualise of the reference (flow_class.py:869-951), for a
// batch of N frames. The one-frame entry points are the N = 1 case of the same kernels.
//
//   magnitude_kernel : mag[n,p] = |threshold(flow[n,p])| exactly as cv2.cartToPolar computes it (float32,
//                      sqrt(fma(x, x, y*y))), the maximum of each frame and, fused, the first histogram pass of the
//                      selection below.
//   hist_kernel /    : exact order statistics of non-negative float32 values by segmented radix selection on the bit
//   pick_kernel        patterns: 3 passes of 12 / 10 / 10 bits, each frame with its own prefixes, ranks and 32-bit
//                      histograms (shared memory per block, one global histogram per frame and rank). One launch per
//                      pass covers all N frames; the bin is chosen on the device. The last pick blends the two order
//                      statistics numpy.percentile(mag, 99) interpolates between and applies the reference's range rule
//                      (99th percentile, else the maximum, else 1): one float per frame, nothing returns to the host.
//   colourise_kernel : hue = cv2's fastAtan2 polynomial (FMA Horner scheme of the AVX2 / AVX-512 code path of the
//                      OpenCV wheels), saturation = clip(mag * 255 / range_max), value 255 (180 on invalid pixels with
//                      show_mask), mask borders = valid pixels with an invalid or out-of-frame 4-neighbour (what
//                      cv2.findContours + drawContours(thickness 1) paint); 'hsv' rounds half-even to uint8, 'rgb' /
//                      'bgr' convert in float64 in numpy's operation order (no contraction: explicit intrinsics).
//                      8 pixels per thread over the flat [N,H,W] index (64-bit), 8-byte stores where aligned.
#include <stddef.h>

#include <algorithm>
#include <cmath>

#include "radix_select.cuh"

namespace ofk {
namespace vis {

__device__ __forceinline__ float thresholded(float c, float thr) { return (c < thr && c > -thr) ? 0.f : c; }

__device__ __forceinline__ float magnitude(float x, float y) { return __fsqrt_rn(__fmaf_rn(x, x, __fmul_rn(y, y))); }

// cv::fastAtan2 in degrees, vector code path (mathfuncs_core.simd.hpp, v_atan_f32): FMA Horner scheme
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
    const float s = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * s, p3 = -0.3258083974640975f * s, p5 = 0.1555786518463281f * s,
                p7 = -0.04432655554792128f * s;
    const float ax = fabsf(x), ay = fabsf(y);
    const float c = __fdiv_rn(fminf(ax, ay), __fadd_rn(fmaxf(ax, ay), 2.220446049250313e-16f));
    const float cc = __fmul_rn(c, c);
    float a = __fmul_rn(__fmaf_rn(__fmaf_rn(__fmaf_rn(cc, p7, p5), cc, p3), cc, p1), c);
    if (!(ax >= ay)) a = __fsub_rn(90.f, a);
    if (x < 0.f) a = __fsub_rn(180.f, a);
    if (y < 0.f) a = __fsub_rn(360.f, a);
    return a;
}

// ------------------------------------------------------------------------------------------------ radix selection
// (digits, histogram helpers: radix_select.cuh)
constexpr int kMaxRanks = 4;

// Per-frame selection record: head, then the histograms (pass 0: one, shared by every rank since no prefix is fixed
// yet; passes 1 and 2: one per rank). Zeroed before the magnitude / first histogram pass.
struct SelectHead {
    unsigned int max_bits;            // maximum magnitude of the frame (bit pattern)
    float range;                      // the frame's range_max, written by the last pick
    unsigned int prefix[kMaxRanks];   // digits found so far
    unsigned int rank[kMaxRanks];     // rank still to resolve among the values with that prefix
};
constexpr size_t kHeadBytes = 256;
static_assert(sizeof(SelectHead) <= kHeadBytes, "SelectHead");

__host__ __device__ constexpr size_t select_frame_bytes(int nq) {
    return kHeadBytes + sizeof(unsigned int) * (kBins0 + 2 * (size_t)nq * kBins12);
}
__host__ __device__ inline unsigned int* pass_hist(char* frame, int pass, int nq, int q) {
    unsigned int* h = reinterpret_cast<unsigned int*>(frame + kHeadBytes);
    if (pass == 0) return h;
    return h + kBins0 + ((size_t)(pass - 1) * nq + q) * kBins12;
}

// Where the selection records of N frames live: frame n at base + n * stride.
struct Select {
    char* base;
    size_t stride;
    int nq;
    __device__ SelectHead* head(size_t n) const { return reinterpret_cast<SelectHead*>(base + n * stride); }
};

constexpr int kUnroll = 4;   // elements per thread and loop trip, strided by the block (coalesced)

// bpf blocks per frame, frame-major on grid x (block b of frame n is blockIdx.x = n * bpf + b: no limit on N but
// grid x's). mag of frame n at mag + n * mag_stride; max_bits at max_base + n * max_stride (uints); sel.base == nullptr:
// no histogram (ofk_vis_magnitude).
__global__ void __launch_bounds__(256) magnitude_kernel(const float2* __restrict__ flow, float thr,
                                                        float* __restrict__ mag, size_t mag_stride, size_t hw,
                                                        unsigned int* __restrict__ max_base, size_t max_stride,
                                                        Select sel, int bpf) {
    __shared__ unsigned int sh[kBins0];
    const bool hist = sel.base != nullptr;
    if (hist) {
        for (int k = threadIdx.x; k < kBins0; k += blockDim.x) sh[k] = 0;
        __syncthreads();
    }
    const size_t n = blockIdx.x / bpf, blk = blockIdx.x - n * bpf;
    const float2* f = flow + n * hw;
    float* m = mag + n * mag_stride;
    unsigned int mx = 0;
    const size_t step = (size_t)bpf * blockDim.x * kUnroll;
    for (size_t base = blk * blockDim.x * kUnroll; base < hw; base += step) {
        float2 v[kUnroll];
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const size_t i = base + j * blockDim.x + threadIdx.x;
            v[j] = i < hw ? __ldg(f + i) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const size_t i = base + j * blockDim.x + threadIdx.x;
            const unsigned int b = __float_as_uint(magnitude(thresholded(v[j].x, thr), thresholded(v[j].y, thr)));
            if (i < hw) {
                m[i] = __uint_as_float(b);
                mx = max(mx, b);
            }
            if (hist) hist_add(sh, b >> 20, i < hw);
        }
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(max_base + n * max_stride, mx);
    if (hist) {
        __syncthreads();
        flush_hist(sh, pass_hist(sel.base + n * sel.stride, 0, sel.nq, 0), kBins0);
    }
}

// One histogram pass of the selection over the values of every frame (bpf blocks per frame on grid x): pass 0 counts
// every value into one histogram, passes 1 and 2 count, per rank, the values whose higher digits equal its prefix.
template <int PASS>
__global__ void __launch_bounds__(256) hist_kernel(const unsigned int* __restrict__ values, size_t stride, size_t n_vals,
                                                   Select sel, int bpf) {
    constexpr int kBins = pass_bins(PASS), kShift = pass_shift(PASS);
    constexpr unsigned int kHiMask = PASS == 0 ? 0u : ~0u << (kShift + 10);
    __shared__ unsigned int sh[PASS == 0 ? kBins0 : kMaxRanks * kBins12];
    const size_t n = blockIdx.x / bpf, blk = blockIdx.x - n * bpf;
    const int nh = PASS == 0 ? 1 : sel.nq;
    for (int k = threadIdx.x; k < nh * kBins; k += blockDim.x) sh[k] = 0;
    unsigned int prefix[kMaxRanks];
    const SelectHead* hd = sel.head(n);
#pragma unroll
    for (int q = 0; q < kMaxRanks; ++q) prefix[q] = q < nh ? hd->prefix[q] : 0u;
    __syncthreads();
    const unsigned int* v = values + n * stride;
    const size_t step = (size_t)bpf * blockDim.x * kUnroll;
    for (size_t base = blk * blockDim.x * kUnroll; base < n_vals; base += step) {
        unsigned int b[kUnroll];
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const size_t i = base + j * blockDim.x + threadIdx.x;
            b[j] = i < n_vals ? __ldg(v + i) : 0u;
        }
#pragma unroll
        for (int j = 0; j < kUnroll; ++j) {
            const bool in = base + j * blockDim.x + threadIdx.x < n_vals;
            const unsigned int bin = (b[j] >> kShift) & (kBins - 1);
            for (int q = 0; q < nh; ++q) {
                const bool hit = in && (b[j] & kHiMask) == prefix[q];
                if (__any_sync(0xffffffffu, hit)) hist_add(sh + q * kBins, bin, hit);
            }
        }
    }
    __syncthreads();
    char* fr = sel.base + n * sel.stride;
    for (int q = 0; q < nh; ++q) flush_hist(sh + q * kBins, pass_hist(fr, PASS, sel.nq, q), kBins);
}

struct Ranks {
    unsigned int r[kMaxRanks];
};

// numpy's _lerp on float32 operands (two-sided, all float32, no contraction)
__device__ __forceinline__ float lerp_np(float a, float b, float gamma) {
    const float d = __fsub_rn(b, a);
    float r = __fadd_rn(a, __fmul_rn(d, gamma));
    if (gamma >= 0.5f) r = __fsub_rn(b, __fmul_rn(d, __fsub_rn(1.f, gamma)));
    return r;
}

// One block per frame: for each rank, the bin of this pass whose cumulative count passes the rank (block-wide scan).
// Pass 0 starts from `ranks`. After pass 2 the prefixes are the values: with out != nullptr they are written to out
// (frame 0 only: ofk_kth_smallest), otherwise ranks 0 / 1 are blended with gamma and the range rule gives head.range.
template <int PASS>
__global__ void __launch_bounds__(256) pick_kernel(Select sel, Ranks ranks, float gamma, float* __restrict__ out) {
    constexpr int kBins = pass_bins(PASS), kShift = pass_shift(PASS), kPer = kBins / 256;
    __shared__ unsigned int warp_sum[8];
    const size_t n = blockIdx.x;
    char* fr = sel.base + n * sel.stride;
    SelectHead* hd = sel.head(n);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int q = 0; q < sel.nq; ++q) {
        const unsigned int* h = pass_hist(fr, PASS, sel.nq, q) + threadIdx.x * kPer;
        const unsigned int rank = PASS == 0 ? ranks.r[q] : hd->rank[q];
        unsigned int c[kPer], local = 0;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            c[k] = h[k];
            local += c[k];
        }
        unsigned int incl = local;   // inclusive scan over the block
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sum[wid] = incl;
        __syncthreads();
        for (int w = 0; w < wid; ++w) incl += warp_sum[w];
        unsigned int excl = incl - local;
        if (excl <= rank && rank < incl) {
            unsigned int r = rank - excl, bin = threadIdx.x * kPer + kPer - 1;
#pragma unroll
            for (int k = 0; k < kPer; ++k) {
                if (r < c[k]) {
                    bin = threadIdx.x * kPer + k;
                    break;
                }
                r -= c[k];
            }
            hd->prefix[q] = (PASS == 0 ? 0u : hd->prefix[q]) | (bin << kShift);
            hd->rank[q] = r;
        }
        __syncthreads();
    }
    if (PASS == 2 && threadIdx.x == 0) {
        if (out != nullptr) {
            for (int q = 0; q < sel.nq; ++q) out[q] = __uint_as_float(hd->prefix[q]);
        } else {
            const float p99 = lerp_np(__uint_as_float(hd->prefix[0]), __uint_as_float(hd->prefix[1]), gamma);
            hd->range = p99 > 0.f ? p99 : (hd->max_bits ? __uint_as_float(hd->max_bits) : 1.f);
        }
    }
}

// ------------------------------------------------------------------------------------------------ colourise
__device__ __forceinline__ uint8_t round_u8(float v) { return (uint8_t)__float2int_rn(v); }   // half-even; 0 <= v <= 255
__device__ __forceinline__ uint8_t round_u8(double v) { return (uint8_t)__double2int_rn(v); }

// One pixel: grey = show_mask and invalid, outline = painted black as part of the mask border.
__device__ __forceinline__ uchar3 colour(float2 f, float thr, float range_max, int mode, bool grey, bool outline) {
    const float fx = thresholded(f.x, thr), fy = thresholded(f.y, thr);
    const float mag = magnitude(fx, fy);
    const float ang = fast_atan2_deg(fy, fx);
    float h = __fmul_rn(ang >= 360.f ? 0.f : ang, 0.5f);                            // np.mod(ang, 360) / 2
    float s = fminf(fmaxf(__fdiv_rn(__fmul_rn(mag, 255.f), range_max), 0.f), 255.f);   // np.clip(mag * 255 / range_max, 0, 255)
    float v = grey ? 180.f : 255.f;
    if (outline) h = s = v = 0.f;
    if (mode == 0) return make_uchar3(round_u8(h), round_u8(s), round_u8(v));
    // hsv -> rgb in numpy's order of operations (flow_class.py:930-945); float32 until `f = h * 6. - i`, float64 after
    // v / 255 for the three values v can take (255 / 255 and 0 / 255 are exact)
    const float vn = outline ? 0.f : (grey ? __fdiv_rn(180.f, 255.f) : 1.f);
    const float hn = __fdiv_rn(h, 180.f), sn = __fdiv_rn(s, 255.f);
    const float h6 = __fmul_rn(hn, 6.f);
    const int i = (int)h6;                                    // np.int_ truncates
    const double fr = __dsub_rn((double)h6, (double)i);
    const double t = __dsub_rn(1.0, fr);
    const double sd = (double)sn, vd = (double)vn;
    const double c0 = __dmul_rn(__dsub_rn(1.0, __dmul_rn(sd, 0.0)), vd);          // v
    const double c1 = __dmul_rn(__dsub_rn(1.0, sd), vd);                          // p  (s * 1)
    const double c2 = __dmul_rn(__dsub_rn(1.0, __dmul_rn(sd, fr)), vd);           // q
    const double c3 = __dmul_rn(__dsub_rn(1.0, __dmul_rn(sd, t)), vd);            // t
    double r, g, b;
    switch (i % 6) {
        case 0: r = c0; g = c3; b = c1; break;
        case 1: r = c2; g = c0; b = c1; break;
        case 2: r = c1; g = c0; b = c3; break;
        case 3: r = c1; g = c2; b = c0; break;
        case 4: r = c3; g = c1; b = c0; break;
        default: r = c0; g = c1; b = c2; break;
    }
    const uint8_t R = round_u8(__dmul_rn(r, 255.0)), G = round_u8(__dmul_rn(g, 255.0)), B = round_u8(__dmul_rn(b, 255.0));
    return mode == 1 ? make_uchar3(R, G, B) : make_uchar3(B, G, R);
}

constexpr int kPx = 8;   // pixels per thread: 64 bytes of flow in, 24 bytes out (three 8-byte stores)

// The range of each frame: range_const, or (range_base != nullptr) the float at range_base + n * range_stride bytes.
struct RangeSrc {
    const char* base;
    size_t stride;
    float value;
    __device__ float of(size_t n) const {
        return base ? *reinterpret_cast<const float*>(base + n * stride) : value;
    }
};

// Flat pixel index p over [N,H,W]; each thread takes kPx consecutive pixels (which may cross rows and frames). vec:
// flow 16-byte, out and mask 8-byte aligned -- then full groups load and store wide, the last group goes pixel by pixel.
__global__ void __launch_bounds__(256) colourise_kernel(const float2* __restrict__ flow,
                                                        const uint8_t* __restrict__ mask, float thr, int mode,
                                                        int show_mask, int show_borders, RangeSrc range,
                                                        uint8_t* __restrict__ out, size_t total, int H, int W,
                                                        int vec) {
    const size_t p0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * kPx;
    if (p0 >= total) return;
    const size_t hw = (size_t)H * W;
    size_t n = p0 / hw;
    const size_t q = p0 - n * hw;
    int y = (int)(q / (size_t)W), x = (int)(q - (size_t)y * W);
    float rmax = range.of(n);
    const bool full = vec && p0 + kPx <= total;
    float2 f[kPx];
    uint8_t mk[kPx];
    if (full) {
        const float4* f4 = reinterpret_cast<const float4*>(flow + p0);
#pragma unroll
        for (int j = 0; j < kPx / 2; ++j) {
            const float4 t = __ldg(f4 + j);   // cached: loads j and j + 1 of a warp share 32-byte sectors
            f[2 * j] = make_float2(t.x, t.y);
            f[2 * j + 1] = make_float2(t.z, t.w);
        }
        if (mask) {
            const uint2 m = __ldg(reinterpret_cast<const uint2*>(mask + p0));
#pragma unroll
            for (int j = 0; j < kPx; ++j) mk[j] = (uint8_t)((j < 4 ? m.x : m.y) >> (8 * (j & 3)));
        }
    } else {
#pragma unroll
        for (int j = 0; j < kPx; ++j) {
            const bool in = p0 + j < total;
            f[j] = in ? __ldg(flow + p0 + j) : make_float2(0.f, 0.f);
            mk[j] = (mask && in) ? __ldg(mask + p0 + j) : 1;
        }
    }
    unsigned long long w[3] = {0ull, 0ull, 0ull};
#pragma unroll
    for (int j = 0; j < kPx; ++j) {
        const size_t p = p0 + j;
        if (!full && p >= total) break;
        const bool valid = mask == nullptr || mk[j] != 0;
        bool outline = false;
        if (show_borders) {
            if (mask == nullptr) {
                outline = y == 0 || y == H - 1 || x == 0 || x == W - 1;
            } else if (valid) {
                const bool inner = y > 0 && y < H - 1 && x > 0 && x < W - 1 && __ldg(mask + p - W) &&
                                   __ldg(mask + p + W) && __ldg(mask + p - 1) && __ldg(mask + p + 1);
                outline = !inner;
            }
        }
        const uchar3 c = colour(f[j], thr, rmax, mode, show_mask && !valid, outline);
        if (full) {
            w[(3 * j) / 8] |= (unsigned long long)c.x << (8 * ((3 * j) % 8));
            w[(3 * j + 1) / 8] |= (unsigned long long)c.y << (8 * ((3 * j + 1) % 8));
            w[(3 * j + 2) / 8] |= (unsigned long long)c.z << (8 * ((3 * j + 2) % 8));
        } else {
            uint8_t* o = out + p * 3;
            o[0] = c.x; o[1] = c.y; o[2] = c.z;
        }
        if (++x == W) {
            x = 0;
            if (++y == H) {
                y = 0;
                ++n;
                if (j + 1 < kPx && p + 1 < total) rmax = range.of(n);
            }
        }
    }
    if (full) {
        unsigned long long* o = reinterpret_cast<unsigned long long*>(out + p0 * 3);
        o[0] = w[0];
        o[1] = w[1];
        o[2] = w[2];
    }
}

// ------------------------------------------------------------------------------------------------ host helpers
// numpy.percentile(a, 99) of n float32 values (method 'linear', numpy 2.x): ranks lo / hi and the weight, all float32
// as numpy computes them for float32 input (numpy/lib/_function_base_impl.py: _QuantileMethods['linear'],
// _get_indexes, _get_gamma). _ops.percentile_plan is the same plan in Python.
struct Plan {
    unsigned int lo, hi;
    float gamma;
};
static Plan percentile_plan(size_t n) {
    volatile float q = 99.f / 100.f;                 // volatile: no excess precision, no contraction
    volatile float vi = (float)(n - 1) * q;
    const float prev = floorf(vi);
    Plan p;
    if (vi >= (float)(n - 1)) {
        p.lo = p.hi = (unsigned int)(n - 1);
    } else {
        p.lo = (unsigned int)prev;
        p.hi = p.lo + 1;
    }
    p.gamma = vi - prev;
    return p;
}

// Blocks per frame of the magnitude / histogram kernels: about 8 blocks per SM over the whole batch, at least one
// per frame, and bpf * frames within grid x (2^31 - 1).
static int blocks_per_frame(size_t n_vals, size_t frames) {
    const size_t want = std::max<size_t>(1, ((size_t)sm_count() * 8 + frames - 1) / frames);
    const size_t most = std::max<size_t>(1, (n_vals + 256 * kUnroll - 1) / (256 * kUnroll));
    return (int)std::min<size_t>(std::min(want, most), std::max<size_t>(1, 0x7fffffffu / frames));
}

// The three histogram / pick passes over values (frame n at values + n * stride), pass 0 optionally fused into the
// magnitude kernel by the caller (fused = true).
static int run_selection(const float* values, size_t stride, size_t n_vals, int N, Select sel, Ranks ranks,
                         float gamma, float* out, bool fused, cudaStream_t st) {
    const int bpf = blocks_per_frame(n_vals, N);
    const unsigned int grid = (unsigned int)bpf * (unsigned int)N;
    const unsigned int* v = reinterpret_cast<const unsigned int*>(values);
    if (!fused) {
        hist_kernel<0><<<grid, 256, 0, st>>>(v, stride, n_vals, sel, bpf);
        OFK_LAUNCHED();
    }
    pick_kernel<0><<<N, 256, 0, st>>>(sel, ranks, gamma, out);
    OFK_LAUNCHED();
    hist_kernel<1><<<grid, 256, 0, st>>>(v, stride, n_vals, sel, bpf);
    OFK_LAUNCHED();
    pick_kernel<1><<<N, 256, 0, st>>>(sel, ranks, gamma, out);
    OFK_LAUNCHED();
    hist_kernel<2><<<grid, 256, 0, st>>>(v, stride, n_vals, sel, bpf);
    OFK_LAUNCHED();
    pick_kernel<2><<<N, 256, 0, st>>>(sel, ranks, gamma, out);
    OFK_LAUNCHED();
    return OFK_OK;
}

static int launch_colourise(const float* flow, const uint8_t* mask, float thr, int mode, int show_mask,
                            int show_borders, RangeSrc range, uint8_t* out, int N, int H, int W, cudaStream_t st) {
    const size_t total = (size_t)N * H * W;
    if (total == 0) return OFK_OK;
    const int vec = aligned16(flow) && (reinterpret_cast<uintptr_t>(out) & 7) == 0 &&
                    (reinterpret_cast<uintptr_t>(mask) & 7) == 0;
    const size_t threads = (total + kPx - 1) / kPx;
    colourise_kernel<<<(unsigned int)((threads + 255) / 256), 256, 0, st>>>(
        reinterpret_cast<const float2*>(flow), mask, thr, mode, show_mask, show_borders, range, out, total, H, W, vec);
    OFK_LAUNCHED();
    return OFK_OK;
}

static size_t pad256(size_t b) { return (b + 255) & ~size_t(255); }
static size_t mag_frame_bytes(int H, int W) { return pad256((size_t)H * W * sizeof(float)); }

}  // namespace vis
}  // namespace ofk

using namespace ofk;

extern "C" int ofk_vis_magnitude(const float* flow, float thr, float* mag, float* max_out, size_t n_pixels,
                                 ofk_stream_t stream) {
    OFK_CHECK_ARG(flow != nullptr && mag != nullptr && max_out != nullptr, "ofk_vis_magnitude: NULL pointer");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(flow) & 7) == 0, "ofk_vis_magnitude: flow must be 8-byte aligned");
    cudaStream_t st = as_stream(stream);
    OFK_CUDA(cudaMemsetAsync(max_out, 0, sizeof(float), st));
    if (n_pixels == 0) return OFK_OK;
    const vis::Select none = {nullptr, 0, 0};
    const int bpf = vis::blocks_per_frame(n_pixels, 1);
    vis::magnitude_kernel<<<bpf, 256, 0, st>>>(reinterpret_cast<const float2*>(flow), thr, mag, 0, n_pixels,
                                               reinterpret_cast<unsigned int*>(max_out), 0, none, bpf);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" size_t ofk_kth_smallest_workspace(int n_ranks) {
    if (n_ranks < 1 || n_ranks > vis::kMaxRanks) return 0;
    return vis::select_frame_bytes(n_ranks);
}

extern "C" int ofk_kth_smallest(const float* values, size_t n, const unsigned long long* ranks_host, int n_ranks,
                                float* out, void* ws, size_t ws_bytes, ofk_stream_t stream) {
    OFK_CHECK_ARG(values != nullptr && out != nullptr && ranks_host != nullptr, "ofk_kth_smallest: NULL pointer");
    OFK_CHECK_ARG(n_ranks >= 1 && n_ranks <= 4, "ofk_kth_smallest: 1 to 4 ranks per call, got %d", n_ranks);
    OFK_CHECK_ARG(n > 0, "ofk_kth_smallest: empty array");
    OFK_CHECK_ARG(n <= 0xffffffffull, "ofk_kth_smallest: at most 2^32 - 1 values (32-bit counts), got %zu", n);
    vis::Ranks ranks = {};
    for (int q = 0; q < n_ranks; ++q) {
        OFK_CHECK_ARG(ranks_host[q] < n, "ofk_kth_smallest: rank %llu out of range (n = %zu)", ranks_host[q], n);
        ranks.r[q] = (unsigned int)ranks_host[q];
    }
    OFK_CHECK_ARG(ws != nullptr && ws_bytes >= ofk_kth_smallest_workspace(n_ranks), "ofk_kth_smallest: workspace too small");
    cudaStream_t st = as_stream(stream);
    const vis::Select sel = {static_cast<char*>(ws), vis::select_frame_bytes(n_ranks), n_ranks};
    OFK_CUDA(cudaMemsetAsync(ws, 0, sel.stride, st));
    return vis::run_selection(values, 0, n, 1, sel, ranks, 0.f, out, false, st);
}

extern "C" int ofk_visualise(const float* flow, const uint8_t* mask, float thr, int mode, int show_mask,
                             int show_mask_borders, float range_max, uint8_t* out, int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(flow != nullptr && out != nullptr, "ofk_visualise: NULL pointer");
    OFK_CHECK_ARG(H > 0 && W > 0, "ofk_visualise: bad shape H=%d W=%d", H, W);
    OFK_CHECK_ARG(mode >= 0 && mode <= 2, "ofk_visualise: mode must be 0 (hsv), 1 (rgb) or 2 (bgr)");
    OFK_CHECK_ARG(range_max > 0.f, "ofk_visualise: range_max must be positive");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(flow) & 7) == 0, "ofk_visualise: flow must be 8-byte aligned");
    const vis::RangeSrc range = {nullptr, 0, range_max};
    return vis::launch_colourise(flow, mask, thr, mode, show_mask, show_mask_borders, range, out, 1, H, W,
                                 as_stream(stream));
}

extern "C" size_t ofk_visualise_batch_workspace(int N, int H, int W) {
    if (N < 0 || H <= 0 || W <= 0) return 0;
    return (size_t)N * (vis::mag_frame_bytes(H, W) + vis::select_frame_bytes(2));
}

extern "C" int ofk_visualise_batch(const float* flow, const uint8_t* mask, float thr, int mode, int show_mask,
                                   int show_mask_borders, float range_max, uint8_t* out, int N, int H, int W, void* ws,
                                   size_t ws_bytes, ofk_stream_t stream) {
    OFK_CHECK_ARG(flow != nullptr && out != nullptr, "ofk_visualise_batch: NULL pointer");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0, "ofk_visualise_batch: bad shape N=%d H=%d W=%d", N, H, W);
    OFK_CHECK_ARG((size_t)H * W < (1ull << 31), "ofk_visualise_batch: a frame needs fewer than 2^31 pixels");
    OFK_CHECK_ARG(mode >= 0 && mode <= 2, "ofk_visualise_batch: mode must be 0 (hsv), 1 (rgb) or 2 (bgr)");
    OFK_CHECK_ARG(range_max >= 0.f, "ofk_visualise_batch: range_max must be positive, or 0 for the default range");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(flow) & 7) == 0, "ofk_visualise_batch: flow must be 8-byte aligned");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 3) == 0, "ofk_visualise_batch: ws must be 4-byte aligned");
    OFK_CHECK_ARG(range_max > 0.f || (ws != nullptr && ws_bytes >= ofk_visualise_batch_workspace(N, H, W)),
                  "ofk_visualise_batch: workspace too small (%zu bytes, need %zu)", ws_bytes,
                  ofk_visualise_batch_workspace(N, H, W));
    if (N == 0) return OFK_OK;
    cudaStream_t st = as_stream(stream);
    if (range_max > 0.f) {
        const vis::RangeSrc range = {nullptr, 0, range_max};
        return vis::launch_colourise(flow, mask, thr, mode, show_mask, show_mask_borders, range, out, N, H, W, st);
    }
    // ws: magnitudes of N frames, then N selection records
    const size_t hw = (size_t)H * W, mag_stride = vis::mag_frame_bytes(H, W) / sizeof(float);
    float* mag = static_cast<float*>(ws);
    const vis::Select sel = {static_cast<char*>(ws) + (size_t)N * vis::mag_frame_bytes(H, W),
                             vis::select_frame_bytes(2), 2};
    OFK_CUDA(cudaMemsetAsync(sel.base, 0, sel.stride * N, st));
    const int bpf = vis::blocks_per_frame(hw, N);
    vis::magnitude_kernel<<<(unsigned int)bpf * (unsigned int)N, 256, 0, st>>>(
        reinterpret_cast<const float2*>(flow), thr, mag, mag_stride, hw,
        reinterpret_cast<unsigned int*>(sel.base + offsetof(vis::SelectHead, max_bits)),
        sel.stride / sizeof(unsigned int), sel, bpf);
    OFK_LAUNCHED();
    const vis::Plan plan = vis::percentile_plan(hw);
    const vis::Ranks ranks = {{plan.lo, plan.hi, 0u, 0u}};
    const int rc = vis::run_selection(mag, mag_stride, hw, N, sel, ranks, plan.gamma, nullptr, true, st);
    if (rc != OFK_OK) return rc;
    const vis::RangeSrc range = {sel.base + offsetof(vis::SelectHead, range), sel.stride, 0.f};
    return vis::launch_colourise(flow, mask, thr, mode, show_mask, show_mask_borders, range, out, N, H, W, st);
}
