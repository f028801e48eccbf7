// Streaming (one-touch) kernels of the flow algebra for sm_100a: Flow.__add__/__sub__/__mul__/... (flow_class.py:310-489),
// the zero / finite tests (flow_class.py:78-79,1230-1245; utils.py:298-316,527-544), Flow.pad (:508-526), the extent
// reduction of get_padding (:1197-1228) and points_inside_area (utils.py:283-295). All HBM-bound; 128-bit accesses,
// grid-stride loops sized to the SM count.
#include <float.h>
#include <math.h>

#include <algorithm>

#include "ofk_common.cuh"
#include "track_device.cuh"

namespace ofk {

static inline int stream_grid(size_t work_items, int threads) {
    size_t blocks = (work_items + threads - 1) / threads;
    size_t cap = (size_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

// ------------------------------------------------------------------------------------------------- add / sub
template <bool SUB>
__global__ void __launch_bounds__(256) addsub_kernel(const float* __restrict__ A, const uint8_t* __restrict__ Am,
                                                     const float* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                     float* __restrict__ out, uint8_t* __restrict__ om, size_t npix,
                                                     int vec_ok) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
    size_t done = 0;
    if (vec_ok) {  // 4 pixels (8 floats, 4 mask bytes) per iteration
        const size_t groups = npix / 4;
        for (size_t g = tid; g < groups; g += nth) {
            const float4* a4 = reinterpret_cast<const float4*>(A) + g * 2;
            const float4* b4 = reinterpret_cast<const float4*>(B) + g * 2;
            float4 a0 = ld_stream_f4(a4), a1 = ld_stream_f4(a4 + 1), b0 = ld_stream_f4(b4), b1 = ld_stream_f4(b4 + 1);
            float4 r0, r1;
            if (SUB) {
                r0 = make_float4(a0.x - b0.x, a0.y - b0.y, a0.z - b0.z, a0.w - b0.w);
                r1 = make_float4(a1.x - b1.x, a1.y - b1.y, a1.z - b1.z, a1.w - b1.w);
            } else {
                r0 = make_float4(a0.x + b0.x, a0.y + b0.y, a0.z + b0.z, a0.w + b0.w);
                r1 = make_float4(a1.x + b1.x, a1.y + b1.y, a1.z + b1.z, a1.w + b1.w);
            }
            float4* o4 = reinterpret_cast<float4*>(out) + g * 2;
            st_stream_f4(o4, r0);
            st_stream_f4(o4 + 1, r1);
            if (om != nullptr) {
                uint32_t ma = Am ? ld_stream_u32(reinterpret_cast<const uint32_t*>(Am) + g) : 0x01010101u;
                uint32_t mb = Bm ? ld_stream_u32(reinterpret_cast<const uint32_t*>(Bm) + g) : 0x01010101u;
                st_stream_u32(reinterpret_cast<uint32_t*>(om) + g, ma & mb);
            }
        }
        done = groups * 4;
    }
    for (size_t i = done + tid; i < npix; i += nth) {
        out[i * 2] = SUB ? A[i * 2] - B[i * 2] : A[i * 2] + B[i * 2];
        out[i * 2 + 1] = SUB ? A[i * 2 + 1] - B[i * 2 + 1] : A[i * 2 + 1] + B[i * 2 + 1];
        if (om != nullptr) om[i] = ((Am ? Am[i] : 1) & (Bm ? Bm[i] : 1)) ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------------- scaling family
template <typename R>
__device__ __forceinline__ R apply_op(int op, R a, R s) {
    switch (op) {
        case OFK_OP_ADD: return a + s;
        case OFK_OP_SUB: return a - s;
        case OFK_OP_MUL: return a * s;
        case OFK_OP_DIV: return a / s;
        default: return pow(a, s);
    }
}

// float32 ** python scalar: numpy sends the exponents 1, -1, 0, 0.5 and 2 to positive / reciprocal / ones_like / sqrt /
// square (fast_scalar_power), all correctly rounded; every other exponent goes to a float32 pow that is not.
__device__ __forceinline__ float pow_f32(float a, float s) {
    if (s == 2.f) return __fmul_rn(a, a);
    if (s == 0.5f) return __fsqrt_rn(a);
    if (s == -1.f) return __fdiv_rn(1.f, a);
    if (s == 1.f) return a;
    if (s == 0.f) return 1.f;
    return powf(a, s);
}

__global__ void __launch_bounds__(256) scale_kernel(int op, const float* __restrict__ A, double su, double sv,
                                                    int in_f64, float* __restrict__ out, size_t npix) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
    const float fu = (float)su, fv = (float)sv;
    for (size_t i = tid; i < npix; i += nth) {
        const float2 a = reinterpret_cast<const float2*>(A)[i];
        float2 r;
        if (in_f64) {
            r.x = (float)apply_op<double>(op, (double)a.x, su);
            r.y = (float)apply_op<double>(op, (double)a.y, sv);
        } else if (op == OFK_OP_POW) {
            r.x = pow_f32(a.x, fu);
            r.y = pow_f32(a.y, fv);
        } else {
            r.x = apply_op<float>(op, a.x, fu);
            r.y = apply_op<float>(op, a.y, fv);
        }
        reinterpret_cast<float2*>(out)[i] = r;
    }
}

__global__ void __launch_bounds__(256) scale_array_kernel(int op, const float* __restrict__ A,
                                                          const double* __restrict__ M, int mc,
                                                          float* __restrict__ out, size_t npix) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
    for (size_t i = tid; i < npix; i += nth) {
        const float2 a = reinterpret_cast<const float2*>(A)[i];
        const double mu = mc == 1 ? M[i] : M[i * 2], mv = mc == 1 ? M[i] : M[i * 2 + 1];
        float2 r;
        r.x = (float)apply_op<double>(op, (double)a.x, mu);
        r.y = (float)apply_op<double>(op, (double)a.y, mv);
        reinterpret_cast<float2*>(out)[i] = r;
    }
}

// ------------------------------------------------------------------------------------------------- reductions
__device__ __forceinline__ bool nz(float c, float thr) { return thr > 0.f ? !(c < thr && c > -thr) : (c != 0.f); }

// combine3_ws.cu: probe + scan zero tests (flags[n] = operand non-zero on a valid pixel)
int launch_c3_zero_flags(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float thr, int* flags,
                         int N, int H, int W, cudaStream_t st);

__global__ void __launch_bounds__(256) finite_kernel(const float* __restrict__ d, size_t n, int* __restrict__ flag) {
    bool bad = false;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        bad |= !isfinite(d[i]);
    if (__syncthreads_or(bad) && threadIdx.x == 0) *flag = 1;
}

// float atomic min/max through the ordered-int trick. The branch is on the sign bit, not on v >= 0: -0.0 is >= 0 but
// as a signed int it is INT_MIN, which would beat every negative value already stored.
__device__ __forceinline__ void atomic_min_f(float* addr, float v) {
    if (__float_as_int(v) >= 0) atomicMin(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f(float* addr, float v) {
    if (__float_as_int(v) >= 0) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
    else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__global__ void extent_init_kernel(float* out4, int N) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) {
        out4[i * 4 + 0] = INFINITY;
        out4[i * 4 + 1] = -INFINITY;
        out4[i * 4 + 2] = INFINITY;
        out4[i * 4 + 3] = -INFINITY;
    }
}

// get_padding: v = threshold(flow); ('s': v *= -1); v[...,0] -= col; v[...,1] -= row; v *= -1  (all float32)
__global__ void __launch_bounds__(256) extent_kernel(const float* __restrict__ F, const uint8_t* __restrict__ M,
                                                     float sign, float thr, float* __restrict__ out4, int H, int W) {
    const int n = blockIdx.y;
    const size_t frame = (size_t)H * W;
    const float2* f = reinterpret_cast<const float2*>(F) + (size_t)n * frame;
    const uint8_t* m = M ? M + (size_t)n * frame : nullptr;
    float mny = INFINITY, mxy = -INFINITY, mnx = INFINITY, mxx = -INFINITY;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < frame; i += (size_t)gridDim.x * blockDim.x) {
        if (m && !m[i]) continue;
        float2 v = f[i];
        if (v.x < thr && v.x > -thr) v.x = 0.f;
        if (v.y < thr && v.y > -thr) v.y = 0.f;
        const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
        const float ex = -(__fsub_rn(sign * v.x, (float)x));
        const float ey = -(__fsub_rn(sign * v.y, (float)y));
        mny = fminf(mny, ey);
        mxy = fmaxf(mxy, ey);
        mnx = fminf(mnx, ex);
        mxx = fmaxf(mxx, ex);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
        mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
        mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
        mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (mny != INFINITY) atomic_min_f(out4 + n * 4 + 0, mny);
        if (mxy != -INFINITY) atomic_max_f(out4 + n * 4 + 1, mxy);
        if (mnx != INFINITY) atomic_min_f(out4 + n * 4 + 2, mnx);
        if (mxx != -INFINITY) atomic_max_f(out4 + n * 4 + 3, mxx);
    }
}

// ------------------------------------------------------------------------------------------------- pad
__device__ __forceinline__ int pad_index(int i, int n, int mode) {  // i relative to the unpadded axis, may be outside
    if ((unsigned)i < (unsigned)n) return i;
    if (mode == OFK_PAD_EDGE) return i < 0 ? 0 : n - 1;
    // numpy 'symmetric': reflect including the edge sample, period 2n
    int p = 2 * n;
    int r = i % p;
    if (r < 0) r += p;
    return r < n ? r : p - 1 - r;
}

__global__ void __launch_bounds__(256) pad_kernel(const float* __restrict__ vecs, const uint8_t* __restrict__ mask,
                                                  float* __restrict__ ov, uint8_t* __restrict__ om, int mode, int H,
                                                  int W, int Ho, int Wo, int top, int left) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int n = blockIdx.z;
    if (x >= Wo || y >= Ho) return;
    const int ys = y - top, xs = x - left;
    const bool inside = (unsigned)ys < (unsigned)H && (unsigned)xs < (unsigned)W;
    const size_t o = ((size_t)n * Ho + y) * Wo + x;
    if (ov != nullptr) {
        float2 v = make_float2(0.f, 0.f);
        if (inside || mode != OFK_PAD_CONSTANT) {
            const int yy = pad_index(ys, H, mode), xx = pad_index(xs, W, mode);
            v = reinterpret_cast<const float2*>(vecs)[((size_t)n * H + yy) * W + xx];
        }
        reinterpret_cast<float2*>(ov)[o] = v;
    }
    if (om != nullptr) om[o] = inside ? (mask ? mask[((size_t)n * H + ys) * W + xs] : 1) : 0;
}

__global__ void __launch_bounds__(256) mask_and_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b,
                                                       uint8_t* __restrict__ out, size_t n, int vec_ok) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
    size_t done = 0;
    if (vec_ok) {
        const size_t words = n / 4;
        for (size_t i = tid; i < words; i += nth)
            reinterpret_cast<uint32_t*>(out)[i] =
                reinterpret_cast<const uint32_t*>(a)[i] & reinterpret_cast<const uint32_t*>(b)[i];
        done = words * 4;
    }
    for (size_t i = done + tid; i < n; i += nth) out[i] = (a[i] & b[i]) ? 1 : 0;
}

// rectangular crop of an [N,H,W] array of `eb`-byte elements to [N,h,w] starting at (y0,x0)
__global__ void __launch_bounds__(256) crop_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int eb,
                                                   int H, int W, int y0, int x0, int h, int w) {
    const int n = blockIdx.z, y = blockIdx.y;
    const size_t row_bytes = (size_t)w * eb;
    const uint8_t* src = in + (((size_t)n * H + y0 + y) * W + x0) * eb;
    uint8_t* dst = out + ((size_t)n * h + y) * row_bytes;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < row_bytes; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// cv2.resize(INTER_LINEAR) of a flow field and its mask (utils.py:493-524, flow_class.py:491-506), bit for bit with
// OpenCV's generic float path (resize.cpp): half-pixel-centre mapping, float32 coefficients, horizontal pass then
// vertical pass, no FMA. Vectors are scaled per axis afterwards; the mask is the resized float mask rounded half-even
// (0.5 -> 0). OpenCV's border rules differ per axis: a column outside [0, W-1] is clamped together with its weight,
// a row outside [0, H-1] only has its index clamped, so a border row is S*(1-fy) + S*fy, which may differ from S.
enum { RESIZE_LINEAR = 0, RESIZE_AREA2 = 1, RESIZE_COPY = 2 };

__device__ __forceinline__ void resize_coord(int d, double scale, int n, bool clamp_weight, int& s0, int& s1,
                                             float& f) {
    float fx = (float)__dadd_rn(__dmul_rn(d + 0.5, scale), -0.5);  // not contracted to an FMA, as in OpenCV
    int sx = (int)floorf(fx);
    fx -= sx;
    if (clamp_weight) {
        if (sx < 0) { fx = 0.f; sx = 0; }
        if (sx >= n - 1) { fx = 0.f; sx = n - 1; }
        s0 = sx;
        s1 = min(sx + 1, n - 1);
    } else {
        s0 = min(max(sx, 0), n - 1);
        s1 = min(max(sx + 1, 0), n - 1);
    }
    f = fx;
}

// One output value from the four taps (00, 01 along x; 10, 11 one row down).
// RESIZE_LINEAR: bilinear blend. RESIZE_AREA2: OpenCV turns INTER_LINEAR at an exact 1/2 x 1/2 scale into INTER_AREA's
// fast path, sum = 0 + (((s00 + s01) + s10) + s11) times 0.25 where the 2x2 block is inside the image; an output whose
// block is cut by the right or bottom edge of an odd-sized input averages the taps it has, summed in the same order.
__device__ __forceinline__ float resize_tap(int mode, float s00, float s01, float s10, float s11, float a0, float a1,
                                            float b0, float b1, bool has_x1, bool has_y1) {
    if (mode == RESIZE_LINEAR) {
        const float r0 = __fadd_rn(__fmul_rn(s00, a0), __fmul_rn(s01, a1));
        const float r1 = __fadd_rn(__fmul_rn(s10, a0), __fmul_rn(s11, a1));
        return __fadd_rn(__fmul_rn(r0, b0), __fmul_rn(r1, b1));
    }
    if (mode == RESIZE_COPY) return s00;
    if (has_x1 && has_y1)
        return __fmul_rn(__fadd_rn(0.f, __fadd_rn(__fadd_rn(__fadd_rn(s00, s01), s10), s11)), 0.25f);
    float sum = __fadd_rn(0.f, s00);
    if (has_x1) sum = __fadd_rn(sum, s01);
    if (has_y1) sum = __fadd_rn(sum, s10);
    return __fdiv_rn(sum, (float)(1 + has_x1 + has_y1));
}

__global__ void __launch_bounds__(256) resize_kernel(const float* __restrict__ vecs, const uint8_t* __restrict__ mask,
                                                     float* __restrict__ ov, uint8_t* __restrict__ om, int H, int W,
                                                     int Ho, int Wo, int mode, double scale_x, double scale_y,
                                                     float mul_u, float mul_v) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    const int n = blockIdx.z;
    if (x >= Wo || y >= Ho) return;
    int x0, x1, y0, y1;
    float fx = 0.f, fy = 0.f;
    bool has_x1 = true, has_y1 = true;
    if (mode == RESIZE_LINEAR) {
        resize_coord(x, scale_x, W, true, x0, x1, fx);
        resize_coord(y, scale_y, H, false, y0, y1, fy);
    } else if (mode == RESIZE_AREA2) {
        x0 = 2 * x;
        y0 = 2 * y;
        has_x1 = x0 + 1 < W;
        has_y1 = y0 + 1 < H;
        x1 = has_x1 ? x0 + 1 : x0;
        y1 = has_y1 ? y0 + 1 : y0;
    } else {
        x0 = x1 = x;
        y0 = y1 = y;
    }
    const float a0 = 1.f - fx, a1 = fx, b0 = 1.f - fy, b1 = fy;
    const size_t fb = (size_t)n * H * W, ob = ((size_t)n * Ho + y) * Wo + x;
    if (ov != nullptr) {
        const float2* f = reinterpret_cast<const float2*>(vecs) + fb;
        const float2 s00 = f[(size_t)y0 * W + x0], s01 = f[(size_t)y0 * W + x1], s10 = f[(size_t)y1 * W + x0],
                     s11 = f[(size_t)y1 * W + x1];
        float2 o;
        o.x = __fmul_rn(resize_tap(mode, s00.x, s01.x, s10.x, s11.x, a0, a1, b0, b1, has_x1, has_y1), mul_u);
        o.y = __fmul_rn(resize_tap(mode, s00.y, s01.y, s10.y, s11.y, a0, a1, b0, b1, has_x1, has_y1), mul_v);
        reinterpret_cast<float2*>(ov)[ob] = o;
    }
    if (om != nullptr) {
        const uint8_t* m = mask + fb;
        const float m00 = m[(size_t)y0 * W + x0], m01 = m[(size_t)y0 * W + x1], m10 = m[(size_t)y1 * W + x0],
                    m11 = m[(size_t)y1 * W + x1];
        const float v = resize_tap(mode, m00, m01, m10, m11, a0, a1, b0, b1, has_x1, has_y1);
        om[ob] = rintf(v) == 1.0f ? 1 : 0;
    }
}

__global__ void __launch_bounds__(256) greater_kernel(const float* __restrict__ v, float thr, uint8_t* __restrict__ out,
                                                      size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = v[i] > thr ? 1 : 0;
}

// Flow vectors at float64 points (row, col) by exact bilinear interpolation (bilinear_track_point); out = pts + (v, u).
// bad[0] is set when a point lies outside [0,H-1]x[0,W-1] (the reference raises IndexError).
__global__ void __launch_bounds__(128) track_bilinear_kernel(const float* __restrict__ flow, const double* __restrict__ pts,
                                                             size_t n, int H, int W, double* __restrict__ out,
                                                             int* __restrict__ bad) {
    const float2* f = reinterpret_cast<const float2*>(flow);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        if (!bilinear_track_point(f, H, W, pts[i * 2], pts[i * 2 + 1], out[i * 2], out[i * 2 + 1])) {
            *bad = 1;
            out[i * 2] = out[i * 2 + 1] = 0.0;
        }
    }
}

__global__ void __launch_bounds__(256) inside_kernel(const double* __restrict__ pts, size_t n, int H, int W,
                                                     uint8_t* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const long long r = __double2ll_rn(pts[i * 2]), c = __double2ll_rn(pts[i * 2 + 1]);  // numpy.round: half-even
        out[i] = (r >= 0 && r <= H - 1 && c >= 0 && c <= W - 1) ? 1 : 0;
    }
}


// ------------------------------------------------------------------------------------------------ dataset decoders
// KITTI flow PNG (utils.py:426-445): uint16 BGR as OpenCV decodes it; u = (R - 2^15) / 64, v = (G - 2^15) / 64 (exact in
// float32), valid = B != 0. Sintel .flo (utils.py:448-471) is little-endian float32 (u, v) already; its invalid-pixel
// PNG (utils.py:474-490) is a uint8 image, valid = (value == 0).
__global__ void __launch_bounds__(256) decode_kitti_kernel(const uint16_t* __restrict__ bgr, float2* __restrict__ vecs,
                                                           uint8_t* __restrict__ mask, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const unsigned b = bgr[3 * i], g = bgr[3 * i + 1], r = bgr[3 * i + 2];
        vecs[i] = make_float2((float)((int)r - 32768) * 0.015625f, (float)((int)g - 32768) * 0.015625f);
        if (mask != nullptr) mask[i] = b != 0 ? 1 : 0;
    }
}
__global__ void __launch_bounds__(256) invert_mask_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out,
                                                          size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = in[i] == 0 ? 1 : 0;
}

}  // namespace ofk

using namespace ofk;

extern "C" int ofk_addsub(int op, const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float* out,
                          uint8_t* out_mask, int N, int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(op == OFK_OP_ADD || op == OFK_OP_SUB, "ofk_addsub: op must be ADD or SUB");
    OFK_CHECK_ARG(A && B && out, "ofk_addsub: NULL operand");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0, "ofk_addsub: bad shape");
    const size_t npix = (size_t)N * H * W;
    if (npix == 0) return OFK_OK;
    const int vec_ok = aligned16(A) && aligned16(B) && aligned16(out) && (!Am || aligned16(Am)) &&
                       (!Bm || aligned16(Bm)) && (!out_mask || aligned16(out_mask));
    const int grid = stream_grid(npix / 4 + 1, 256);
    if (op == OFK_OP_SUB)
        addsub_kernel<true><<<grid, 256, 0, as_stream(stream)>>>(A, Am, B, Bm, out, out_mask, npix, vec_ok);
    else
        addsub_kernel<false><<<grid, 256, 0, as_stream(stream)>>>(A, Am, B, Bm, out, out_mask, npix, vec_ok);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_scale(int op, const float* A, double su, double sv, int in_f64, float* out, size_t n_pixels,
                         ofk_stream_t stream) {
    OFK_CHECK_ARG(op >= OFK_OP_MUL && op <= OFK_OP_POW, "ofk_scale: op must be MUL, DIV or POW");
    OFK_CHECK_ARG(A && out, "ofk_scale: NULL operand");
    OFK_CHECK_ARG(((uintptr_t)A & 7) == 0 && ((uintptr_t)out & 7) == 0, "ofk_scale: pointers must be 8-byte aligned");
    if (n_pixels == 0) return OFK_OK;
    scale_kernel<<<stream_grid(n_pixels, 256), 256, 0, as_stream(stream)>>>(op, A, su, sv, in_f64, out, n_pixels);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_scale_array(int op, const float* A, const double* M, int m_channels, float* out, size_t n_pixels,
                               ofk_stream_t stream) {
    OFK_CHECK_ARG(op >= OFK_OP_ADD && op <= OFK_OP_POW, "ofk_scale_array: unknown op %d", op);
    OFK_CHECK_ARG(A && M && out, "ofk_scale_array: NULL operand");
    OFK_CHECK_ARG(m_channels == 1 || m_channels == 2, "ofk_scale_array: m_channels must be 1 or 2");
    OFK_CHECK_ARG(((uintptr_t)A & 7) == 0 && ((uintptr_t)out & 7) == 0, "ofk_scale_array: pointers must be 8-byte aligned");
    if (n_pixels == 0) return OFK_OK;
    scale_array_kernel<<<stream_grid(n_pixels, 256), 256, 0, as_stream(stream)>>>(op, A, M, m_channels, out, n_pixels);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_nonzero_flags(const float* F, const uint8_t* M, float thr, int* flags, int N, int H, int W,
                                 ofk_stream_t stream) {
    OFK_CHECK_ARG(F && flags, "ofk_nonzero_flags: NULL argument");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0 && N <= 65535, "ofk_nonzero_flags: bad shape");
    OFK_CHECK_ARG(((uintptr_t)F & 7) == 0, "ofk_nonzero_flags: F must be 8-byte aligned");
    if (N == 0) return OFK_OK;
    // a sparse probe proves "not zero" for almost every real flow without reading it; only frames the probe leaves
    // undecided are scanned completely (combine3_ws.cu)
    return launch_c3_zero_flags(F, M, nullptr, nullptr, thr, flags, N, H, W, as_stream(stream));
}

extern "C" int ofk_check_finite(const float* data, size_t n, int* flag, ofk_stream_t stream) {
    OFK_CHECK_ARG(data && flag, "ofk_check_finite: NULL argument");
    cudaStream_t st = as_stream(stream);
    OFK_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    if (n == 0) return OFK_OK;
    finite_kernel<<<stream_grid(n / 4 + 1, 256), 256, 0, st>>>(data, n, flag);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_pad(const float* vecs, const uint8_t* mask, float* out_vecs, uint8_t* out_mask, int mode, int N,
                       int H, int W, int top, int bottom, int left, int right, ofk_stream_t stream) {
    OFK_CHECK_ARG(mode >= OFK_PAD_CONSTANT && mode <= OFK_PAD_SYMMETRIC, "ofk_pad: unknown mode %d", mode);
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0 && top >= 0 && bottom >= 0 && left >= 0 && right >= 0, "ofk_pad: bad shape");
    OFK_CHECK_ARG((out_vecs == nullptr) || vecs != nullptr, "ofk_pad: out_vecs given without vecs");
    OFK_CHECK_ARG(out_vecs != nullptr || out_mask != nullptr, "ofk_pad: nothing to do");
    OFK_CHECK_ARG(!out_vecs || ((((uintptr_t)vecs | (uintptr_t)out_vecs) & 7) == 0), "ofk_pad: vecs must be 8-byte aligned");
    if (N == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_pad: N too large");
    const int Ho = H + top + bottom, Wo = W + left + right;
    dim3 grid((Wo + 31) / 32, (Ho + 7) / 8, N);
    pad_kernel<<<grid, 256, 0, as_stream(stream)>>>(vecs, mask, out_vecs, out_mask, mode, H, W, Ho, Wo, top, left);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_extent(const float* flow, const uint8_t* mask, float sign, float thr, float* out4, int N, int H,
                          int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(flow && out4, "ofk_extent: NULL argument");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0 && N <= 65535, "ofk_extent: bad shape");
    OFK_CHECK_ARG(((uintptr_t)flow & 7) == 0, "ofk_extent: flow must be 8-byte aligned");
    if (N == 0) return OFK_OK;
    cudaStream_t st = as_stream(stream);
    extent_init_kernel<<<(N + 255) / 256, 256, 0, st>>>(out4, N);
    OFK_LAUNCHED();
    const size_t frame = (size_t)H * W;
    int bx = (int)((frame + 256 * 8 - 1) / (256 * 8));
    const int cap = (sm_count() * 8 + N - 1) / N;
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    extent_kernel<<<dim3(bx, N), 256, 0, st>>>(flow, mask, sign, thr, out4, H, W);
    OFK_LAUNCHED();
    return OFK_OK;
}

// dtype conversion of payloads around the float32 forward resampler (utils.py:256-258: np.round for integer targets,
// then astype): to float32 exact for the 8 / 16-bit types; from float32 with round-half-even and saturation.
namespace ofk {
template <class T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ uint8_t from_f32<uint8_t>(float v) {
    return (uint8_t)min(255, max(0, __float2int_rn(v)));
}
template <>
__device__ __forceinline__ int16_t from_f32<int16_t>(float v) {
    return (int16_t)min(32767, max(-32768, __float2int_rn(v)));
}
template <>
__device__ __forceinline__ uint16_t from_f32<uint16_t>(float v) {
    return (uint16_t)min(65535, max(0, __float2int_rn(v)));
}
template <>
__device__ __forceinline__ double from_f32<double>(float v) {
    return (double)v;
}
template <class T>
__global__ void __launch_bounds__(256) cast_to_f32_kernel(const T* __restrict__ in, float* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) out[i] = (float)in[i];
}
template <class T>
__global__ void __launch_bounds__(256) cast_from_f32_kernel(const float* __restrict__ in, T* __restrict__ out,
                                                            size_t n) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256)
        out[i] = from_f32<T>(in[i]);
}
}  // namespace ofk

extern "C" int ofk_cast(const void* in, int in_dtype, void* out, int out_dtype, size_t n, ofk_stream_t stream) {
    OFK_CHECK_ARG(in && out, "ofk_cast: NULL argument");
    OFK_CHECK_ARG((in_dtype == OFK_F32) != (out_dtype == OFK_F32), "ofk_cast: exactly one side must be float32");
    if (n == 0) return OFK_OK;
    cudaStream_t st = as_stream(stream);
    const unsigned grid = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)sm_count() * 16);
    const int other = in_dtype == OFK_F32 ? out_dtype : in_dtype;
    OFK_CHECK_ARG(other == OFK_U8 || other == OFK_I16 || other == OFK_U16 || other == OFK_F64, "ofk_cast: bad dtype %d",
                  other);
#define OFK_CAST(T)                                                                                               \
    do {                                                                                                          \
        if (out_dtype == OFK_F32) cast_to_f32_kernel<T><<<grid, 256, 0, st>>>((const T*)in, (float*)out, n);      \
        else cast_from_f32_kernel<T><<<grid, 256, 0, st>>>((const float*)in, (T*)out, n);                         \
    } while (0)
    switch (other) {
        case OFK_U8: OFK_CAST(uint8_t); break;
        case OFK_I16: OFK_CAST(int16_t); break;
        case OFK_U16: OFK_CAST(uint16_t); break;
        default: OFK_CAST(double); break;
    }
#undef OFK_CAST
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_mask_and(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, ofk_stream_t stream) {
    OFK_CHECK_ARG(a && b && out, "ofk_mask_and: NULL argument");
    if (n == 0) return OFK_OK;
    const int vec_ok = (((uintptr_t)a | (uintptr_t)b | (uintptr_t)out) & 3) == 0;
    mask_and_kernel<<<stream_grid(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(a, b, out, n, vec_ok);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_crop(const void* in, void* out, int elem_bytes, int N, int H, int W, int y0, int x0, int h, int w,
                        ofk_stream_t stream) {
    OFK_CHECK_ARG(in && out && elem_bytes > 0, "ofk_crop: bad argument");
    OFK_CHECK_ARG(N >= 0 && y0 >= 0 && x0 >= 0 && h > 0 && w > 0 && y0 + h <= H && x0 + w <= W && h <= 65535 &&
                      N <= 65535,
                  "ofk_crop: window (%d,%d)+(%d,%d) outside (%d,%d)", y0, x0, h, w, H, W);
    if (N == 0) return OFK_OK;
    int bx = (int)(((size_t)w * elem_bytes + 255) / 256);
    if (bx > 8) bx = 8;
    crop_kernel<<<dim3(bx, h, N), 256, 0, as_stream(stream)>>>((const uint8_t*)in, (uint8_t*)out, elem_bytes, H, W, y0,
                                                              x0, h, w);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_resize_flow(const float* vecs, const uint8_t* mask, float* out_vecs, uint8_t* out_mask, int N, int H,
                               int W, int Ho, int Wo, double fy, double fx, ofk_stream_t stream) {
    OFK_CHECK_ARG((vecs && out_vecs) || (mask && out_mask), "ofk_resize_flow: nothing to do");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0 && Ho > 0 && Wo > 0 && fx > 0 && fy > 0, "ofk_resize_flow: bad shape / scale");
    OFK_CHECK_ARG(!out_vecs || ((((uintptr_t)vecs | (uintptr_t)out_vecs) & 7) == 0), "ofk_resize_flow: vecs must be 8-byte aligned");
    if (N == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_resize_flow: N too large");
    // cv::resize: an output of the input's size is a copy; INTER_LINEAR at an inverse scale of exactly 2 on both axes
    // (|1/f - 2| < DBL_EPSILON) is INTER_AREA's fast path
    const double sx = 1.0 / fx, sy = 1.0 / fy;
    const int mode = (Ho == H && Wo == W)                                           ? RESIZE_COPY
                     : (fabs(sx - 2.0) < DBL_EPSILON && fabs(sy - 2.0) < DBL_EPSILON) ? RESIZE_AREA2
                                                                                      : RESIZE_LINEAR;
    dim3 grid((Wo + 31) / 32, (Ho + 7) / 8, N);
    resize_kernel<<<grid, 256, 0, as_stream(stream)>>>(out_vecs ? vecs : nullptr, out_mask ? mask : nullptr, out_vecs,
                                                      out_mask, H, W, Ho, Wo, mode, sx, sy, (float)fx, (float)fy);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_greater(const float* v, float thr, uint8_t* out, size_t n, ofk_stream_t stream) {
    OFK_CHECK_ARG(v && out, "ofk_greater: NULL argument");
    if (n == 0) return OFK_OK;
    greater_kernel<<<stream_grid(n, 256), 256, 0, as_stream(stream)>>>(v, thr, out, n);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_track_bilinear(const float* flow, const double* pts, size_t n, int H, int W, double* out, int* bad,
                                  ofk_stream_t stream) {
    OFK_CHECK_ARG(flow && pts && out && bad, "ofk_track_bilinear: NULL argument");
    OFK_CHECK_ARG(H > 0 && W > 0, "ofk_track_bilinear: bad shape");
    cudaStream_t st = as_stream(stream);
    OFK_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), st));
    if (n == 0) return OFK_OK;
    track_bilinear_kernel<<<stream_grid(n, 128), 128, 0, st>>>(flow, pts, n, H, W, out, bad);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_points_inside_area(const double* pts, size_t n, int H, int W, uint8_t* out, ofk_stream_t stream) {
    OFK_CHECK_ARG(pts && out, "ofk_points_inside_area: NULL argument");
    if (n == 0) return OFK_OK;
    inside_kernel<<<stream_grid(n, 256), 256, 0, as_stream(stream)>>>(pts, n, H, W, out);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_decode_kitti(const uint16_t* bgr, float* vecs, uint8_t* mask, size_t n_pixels, ofk_stream_t stream) {
    OFK_CHECK_ARG(bgr && vecs, "ofk_decode_kitti: NULL argument");
    OFK_CHECK_ARG(((uintptr_t)vecs & 7) == 0 && ((uintptr_t)bgr & 1) == 0, "ofk_decode_kitti: misaligned pointer");
    if (n_pixels == 0) return OFK_OK;
    decode_kitti_kernel<<<stream_grid(n_pixels, 256), 256, 0, as_stream(stream)>>>(bgr, reinterpret_cast<float2*>(vecs),
                                                                                  mask, n_pixels);
    OFK_LAUNCHED();
    return OFK_OK;
}

extern "C" int ofk_decode_sintel_mask(const uint8_t* invalid, uint8_t* mask, size_t n_pixels, ofk_stream_t stream) {
    OFK_CHECK_ARG(invalid && mask, "ofk_decode_sintel_mask: NULL argument");
    if (n_pixels == 0) return OFK_OK;
    invert_mask_kernel<<<stream_grid(n_pixels, 256), 256, 0, as_stream(stream)>>>(invalid, mask, n_pixels);
    OFK_LAUNCHED();
    return OFK_OK;
}
