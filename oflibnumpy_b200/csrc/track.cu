// Batched point tracking, ofk_track: Flow.track (flow_class.py:755-795, utils.py:547-622) of N frames in one launch.
// The 's' lookup kernel lives here; the mesh route ('t', 's' exact with float points) is next to ofk_mesh_sample in
// forward_s.cu. Both fold the frame into a flat [N*P] point index and share the per-point arithmetic of
// track_device.cuh.
// Trajectories through clips, ofk_track_clips: the entry point and its checks are here, the kernel (which needs the
// mesh) is next to the mesh kernel in forward_s.cu.
#include <limits.h>

#include <algorithm>

#include "track_device.cuh"

namespace ofk {

// ref 's' lookup, one thread per point: integer points (in any mode) index the flow like numpy (an index in [-H,-1]
// wraps) and add the vector in the arithmetic type AT (numpy's result type of pts + float32); float points (without
// exact mode) interpolate it bilinearly in float64 (bilinear_track_point).
template <typename PT, typename AT>
__global__ void __launch_bounds__(256) track_s_kernel(const float2* __restrict__ flow, const uint8_t* __restrict__ mask,
                                                      const int* __restrict__ flow_nonzero, const PT* __restrict__ pts,
                                                      int pts_shared, int P, void* __restrict__ out, int int_out,
                                                      uint8_t* __restrict__ status, int* __restrict__ errors, int H,
                                                      int W, size_t total) {
    const size_t hw = (size_t)H * W;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (size_t)gridDim.x * blockDim.x) {
        const size_t n = k / (size_t)P;
        const size_t i = pts_shared ? k - n * P : k;
        const PT r = pts[2 * i], c = pts[2 * i + 1];
        const float2* f = flow + n * hw;
        int err = 0;
        if (flow_nonzero[n] == 0) {
            store_passthrough<PT, AT>(out, int_out, k, r, c);
        } else if constexpr (std::is_integral<PT>::value) {
            AT orow = 0, ocol = 0;
            if (r < -H || r >= H || c < -W || c >= W) {
                err |= OFK_TRACK_ERR_INDEX;
            } else {
                const float2 d = f[(size_t)(r < 0 ? r + H : r) * W + (size_t)(c < 0 ? c + W : c)];
                if constexpr (std::is_same<AT, float>::value) {
                    orow = __fadd_rn((float)r, d.y);
                    ocol = __fadd_rn((float)c, d.x);
                } else {
                    orow = __dadd_rn((double)r, (double)d.y);
                    ocol = __dadd_rn((double)c, (double)d.x);
                }
            }
            store_tracked<AT>(out, int_out, k, orow, ocol);
        } else {
            double orow = 0.0, ocol = 0.0;
            if (!bilinear_track_point(f, H, W, (double)r, (double)c, orow, ocol)) err |= OFK_TRACK_ERR_OUTSIDE;
            store_tracked<double>(out, int_out, k, orow, ocol);
        }
        if (status != nullptr) track_status(r, c, f, mask ? mask + n * hw : nullptr, nullptr, H, W, k, status, err);
        if (err) atomicOr(errors + n, err);
    }
}

template <typename PT, typename AT>
static int launch_track_s(const float* flow, const uint8_t* mask, const int* flow_nonzero, const void* pts,
                          int pts_shared, int P, void* out, int int_out, uint8_t* status, int* errors, int N, int H,
                          int W, cudaStream_t st) {
    const size_t total = (size_t)N * P;
    const size_t blocks = std::min((total + 255) / 256, (size_t)sm_count() * 32);
    track_s_kernel<PT, AT><<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float2*>(flow), mask, flow_nonzero,
                                                             static_cast<const PT*>(pts), pts_shared, P, out, int_out,
                                                             status, errors, H, W, total);
    OFK_LAUNCHED();
    return OFK_OK;
}

}  // namespace ofk

using namespace ofk;

extern "C" int ofk_track(const float* flow, const uint8_t* mask, int ref, int exact, const int* flow_nonzero,
                         const void* pts, int pts_dtype, int pts_shared, int P, int arith, int int_out, void* out,
                         const uint8_t* status_plane, uint8_t* status, int* errors, int N, int H, int W,
                         ofk_stream_t stream) {
    OFK_CHECK_ARG(flow && flow_nonzero && pts && out && errors, "ofk_track: NULL pointer");
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofk_track: ref must be 's' or 't'");
    OFK_CHECK_ARG(pts_dtype == OFK_F32 || pts_dtype == OFK_F64 || pts_dtype == OFK_I32 || pts_dtype == OFK_I64,
                  "ofk_track: pts_dtype must be OFK_F32, OFK_F64, OFK_I32 or OFK_I64");
    OFK_CHECK_ARG(arith == OFK_F32 || arith == OFK_F64, "ofk_track: arith must be OFK_F32 or OFK_F64");
    OFK_CHECK_ARG(N >= 0 && P >= 0 && H > 0 && W > 0, "ofk_track: bad shape N=%d P=%d H=%d W=%d", N, P, H, W);
    const bool int_pts = pts_dtype == OFK_I32 || pts_dtype == OFK_I64;
    const bool mesh = ref == 't' || (exact != 0 && !int_pts);      // Flow.track looks integer points up on 's' flows
    OFK_CHECK_ARG(arith == OFK_F64 || (int_pts && ref == 's'),
                  "ofk_track: float32 arithmetic needs integer points on an 's' flow");
    OFK_CHECK_ARG(!mesh || (H > 1 && W > 1 && (size_t)H * W < ((size_t)1 << 30)),
                  "ofk_track: the mesh route needs 2 <= H, W and H*W < 2^30 (H=%d W=%d)", H, W);
    OFK_CHECK_ARG(status == nullptr || ref == 's' || status_plane != nullptr,
                  "ofk_track: ref 't' status needs status_plane");
    if (N == 0) return OFK_OK;
    cudaStream_t st = as_stream(stream);
    OFK_CUDA(cudaMemsetAsync(errors, 0, sizeof(int) * (size_t)N, st));
    if (P == 0) return OFK_OK;
    int_out = int_out != 0;
    if (mesh)
        return launch_track_mesh(flow, mask, ref, flow_nonzero, pts, pts_dtype, pts_shared, P, out, int_out,
                                 ref == 't' ? status_plane : nullptr, status, errors, N, H, W, st);
#define OFK_TRACK_S(PT, AT) \
    return launch_track_s<PT, AT>(flow, mask, flow_nonzero, pts, pts_shared, P, out, int_out, status, errors, N, H, W, st)
    switch (pts_dtype) {
        case OFK_F32: OFK_TRACK_S(float, double);
        case OFK_F64: OFK_TRACK_S(double, double);
        case OFK_I32:
            if (arith == OFK_F32) OFK_TRACK_S(int32_t, float);
            OFK_TRACK_S(int32_t, double);
        default:
            if (arith == OFK_F32) OFK_TRACK_S(int64_t, float);
            OFK_TRACK_S(int64_t, double);
    }
#undef OFK_TRACK_S
}

extern "C" int ofk_track_clips(const float* flow, const uint8_t* mask, int ref, int exact, const int* flow_nonzero,
                               const void* pts, int pts_dtype, int pts_shared, int S, int L, int P,
                               const uint8_t* keep, double* out, uint8_t* alive, int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(flow && flow_nonzero && pts && out && alive, "ofk_track_clips: NULL pointer");
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofk_track_clips: ref must be 's' or 't'");
    OFK_CHECK_ARG(pts_dtype == OFK_F32 || pts_dtype == OFK_F64, "ofk_track_clips: pts_dtype must be OFK_F32 or OFK_F64");
    OFK_CHECK_ARG(S >= 0 && L > 0 && P >= 0 && H > 0 && W > 0, "ofk_track_clips: bad shape S=%d L=%d P=%d H=%d W=%d", S,
                  L, P, H, W);
    OFK_CHECK_ARG((long long)S * L <= INT_MAX, "ofk_track_clips: S*L must not exceed INT_MAX (S=%d L=%d)", S, L);
    const bool mesh = ref == 't' || exact != 0;
    OFK_CHECK_ARG(!mesh || (H > 1 && W > 1 && (size_t)H * W < ((size_t)1 << 30)),
                  "ofk_track_clips: the mesh route needs 2 <= H, W and H*W < 2^30 (H=%d W=%d)", H, W);
    if (S == 0 || P == 0) return OFK_OK;
    return launch_track_clips(flow, mask, ref, exact, flow_nonzero, pts, pts_dtype, pts_shared, S, L, P, keep, out,
                              alive, H, W, as_stream(stream));
}
