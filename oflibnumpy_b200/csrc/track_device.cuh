// Per-point arithmetic of point tracking (Flow.track, utils.py:547-622), shared by ofk_track_bilinear (elementwise.cu),
// the lookup kernel of ofk_track (track.cu) and its mesh kernel (forward_s.cu).
#pragma once
#include <math.h>

#include <type_traits>

#include "ofk_common.cuh"

// error bits of ofk_track, one int32 word per frame
#define OFK_TRACK_ERR_OUTSIDE 1   // a float point on an 's' flow outside [0,H-1]x[0,W-1]
#define OFK_TRACK_ERR_INDEX 2     // an integer point on an 's' flow outside [-H,H-1]x[-W,W-1]
#define OFK_TRACK_ERR_STATUS 4    // a rounded point outside [-H,H-1]x[-W,W-1] (get_valid_status)

namespace ofk {

#ifdef __CUDACC__

// Flow vector at the float64 point (r, c) by exact bilinear interpolation with clipped neighbours, float64 arithmetic in
// the reference's operation order (utils.py:161-196); returns false (and leaves the outputs alone) when the point lies
// outside [0,H-1]x[0,W-1], where the reference raises IndexError. f is one frame [H,W] of (u, v).
__device__ __forceinline__ bool bilinear_track_point(const float2* __restrict__ f, int H, int W, double r, double c,
                                                     double& out_r, double& out_c) {
    if (!(0 <= r && r <= H - 1) || !(0 <= c && c <= W - 1)) return false;
    const int r0 = (int)floor(r), c0 = (int)floor(c);
    const int r0c = min(max(r0, 0), H - 1), c0c = min(max(c0, 0), W - 1);
    const int r1c = min(max(r0 + 1, 0), H - 1), c1c = min(max(c0 + 1, 0), W - 1);
    const double wa = __dmul_rn((double)r1c - r, (double)c1c - c), wb = __dmul_rn((double)r1c - r, c - (double)c0c);
    const double wc = __dmul_rn(r - (double)r0c, (double)c1c - c), wd = __dmul_rn(r - (double)r0c, c - (double)c0c);
    const float2 a = f[(size_t)r0c * W + c0c], b = f[(size_t)r1c * W + c0c], cc = f[(size_t)r0c * W + c1c],
                 d = f[(size_t)r1c * W + c1c];
    // result = wa*data_a + wb*data_b + wc*data_c + wd*data_d, data in (v, u) order, no FMA contraction
    const double dv = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(wa, (double)a.y), __dmul_rn(wb, (double)b.y)),
                                          __dmul_rn(wc, (double)cc.y)), __dmul_rn(wd, (double)d.y));
    const double du = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(wa, (double)a.x), __dmul_rn(wb, (double)b.x)),
                                          __dmul_rn(wc, (double)cc.x)), __dmul_rn(wd, (double)d.x));
    out_r = __dadd_rn(r, dv);
    out_c = __dadd_rn(c, du);
    return true;
}

// numpy's `np.round(x).astype('i')` for float64 x on x86-64: round half to even, and INT_MIN (the conversion's
// "integer indefinite") for NaN and values outside the int32 range.
__device__ __forceinline__ int round_to_i32(double x) {
    const double r = rint(x);
    return (r >= -2147483648.0 && r <= 2147483647.0) ? (int)r : (-2147483647 - 1);
}

// The index `np.round(pts).astype('i')` that Flow.track's status reads: integer points are truncated to int32 (the
// cast wraps, as numpy's does), float points rounded half to even.
template <typename PT>
__device__ __forceinline__ int status_index(PT v) {
    if constexpr (std::is_integral<PT>::value) return (int)v;
    else return round_to_i32((double)v);
}

// Frame-wise valid_source of an 's' flow at pixel (y, x): the per-pixel test of valid_geom_vec4 (warp_t.cu) with sign +1.
__device__ __forceinline__ uint8_t valid_source_s_at(const float2* __restrict__ f, const uint8_t* __restrict__ mask,
                                                     int H, int W, int y, int x) {
    const size_t q = (size_t)y * W + x;
    const float2 v = f[q];
    const unsigned ok = strict_in_frame(__fmaf_rn(1.0f, v.x, (float)x), __fmaf_rn(1.0f, v.y, (float)y), H, W);
    return (uint8_t)(ok & (mask ? (unsigned)mask[q] : 1u));
}

// The valid status of one point at its rounded position (ref 's': computed here from flow and mask; ref 't': gathered
// from status_plane) and the error bit when that index is out of range. f, mask and status_plane point at the frame.
template <typename PT>
__device__ __forceinline__ void track_status(PT r, PT c, const float2* __restrict__ f, const uint8_t* __restrict__ mask,
                                             const uint8_t* __restrict__ status_plane, int H, int W, size_t k,
                                             uint8_t* __restrict__ status, int& err) {
    int y = status_index(r), x = status_index(c);
    uint8_t s = 0;
    if (y < -H || y >= H || x < -W || x >= W) {
        err |= OFK_TRACK_ERR_STATUS;
    } else {
        y += y < 0 ? H : 0;
        x += x < 0 ? W : 0;
        s = status_plane ? status_plane[(size_t)y * W + x] : valid_source_s_at(f, mask, H, W, y, x);
    }
    status[k] = s;
}

// Stores a tracked point (row, col) of arithmetic type AT (float or double) as AT or, with int_out, as
// np.round(...).astype('i') of it.
template <typename AT>
__device__ __forceinline__ void store_tracked(void* out, int int_out, size_t k, AT r, AT c) {
    if (int_out) {
        int* o = static_cast<int*>(out) + 2 * k;
        o[0] = round_to_i32((double)r);
        o[1] = round_to_i32((double)c);
    } else {
        AT* o = static_cast<AT*>(out) + 2 * k;
        o[0] = r;
        o[1] = c;
    }
}

// A point of a frame whose flow is zero below the threshold: Flow.track hands the points back, so they are stored
// converted to the batch's output type (with int_out, `np.round(pts).astype('i')`, which truncates integers to int32).
template <typename PT, typename AT>
__device__ __forceinline__ void store_passthrough(void* out, int int_out, size_t k, PT r, PT c) {
    if (int_out && std::is_integral<PT>::value) {
        int* o = static_cast<int*>(out) + 2 * k;
        o[0] = (int)r;
        o[1] = (int)c;
    } else {
        store_tracked<AT>(out, int_out, k, (AT)r, (AT)c);
    }
}

#endif  // __CUDACC__

// ofk_track's mesh route ('t', and 's' with exact = 1), forward_s.cu; arguments checked by the caller
int launch_track_mesh(const float* flow, const uint8_t* mask, int ref, const int* flow_nonzero, const void* pts,
                      int pts_dtype, int pts_shared, int P, void* out, int int_out, const uint8_t* status_plane,
                      uint8_t* status, int* errors, int N, int H, int W, cudaStream_t st);

}  // namespace ofk
