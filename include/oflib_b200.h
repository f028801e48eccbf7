/*
 * oflib_b200 -- C ABI of the B200-native flow-field hot path (drop-in boundary for oflibnumpy's hot path).
 *
 * The reference (oflibnumpy v1.1.1) is pure Python: its "FFI" for this path is the set of call sites where its
 * Python code enters third-party native code, plus the numpy array expressions around them. Each entry point below
 * names the reference interface it replaces (file:line under /root/reference/src/oflibnumpy/). INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add at those call sites.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++/torch types.
 *   - ofk_*  : device pointers owned by the caller, outputs pre-allocated by the caller, asynchronous on `stream`
 *              (a cudaStream_t passed as void*; NULL = legacy default stream). No allocation inside unless a
 *              workspace argument says so.
 *   - ofh_*  : host pointers (numpy buffers, pinned or pageable); the library stages them through an internal
 *              pinned/device ring and overlaps H2D, kernels and D2H. Synchronous: results are in the output buffers
 *              on return.
 *   - ofk_rt_*: the minimal runtime the Python shim needs (memory, streams, events); thin cudart wrappers.
 *   - every function returns 0 on success or a negative OFK_E* code; ofk_last_error() returns a thread-local message.
 *   - layouts are the reference's: flow vectors float32 [N,H,W,2] (channel 0 = horizontal u, +right; 1 = vertical v,
 *     +down; flow_class.py:42-44), masks uint8 0/1 [N,H,W] (numpy bool), images [N,H,W,C] interleaved. N is the batch
 *     axis this library adds (the reference has none; N = 1 reproduces it).
 *   - base pointers should be 16-byte aligned (cudaMalloc / torch allocations are); unaligned pointers are accepted and
 *     take a slower scalar path.
 */
#ifndef OFLIB_B200_H
#define OFLIB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden; these are its exports */
#endif

#define OFK_VERSION 100

/* error codes */
#define OFK_OK 0
#define OFK_EINVAL (-1)   /* bad argument (shape, enum, NULL) */
#define OFK_ECUDA (-2)    /* CUDA runtime error, see ofk_last_error() */
#define OFK_ENOMEM (-3)
#define OFK_EUNSUPPORTED (-4)

/* payload element types accepted by the warp (the dtypes cv2.remap accepts for the reference's calls) */
#define OFK_U8 0
#define OFK_I16 1
#define OFK_U16 2
#define OFK_F32 3
#define OFK_F64 4
/* point element types of ofk_track (besides OFK_F32 / OFK_F64) */
#define OFK_I32 5
#define OFK_I64 6

/* interpolation arithmetic (OpenCV picks it from the dtype of the array handed to cv2.remap, which for Flow.apply is
 * the numpy promotion of payload||mask -- flow_class.py:615,644):
 *   NATIVE : by payload dtype: U8 -> 15-bit fixed point; I16/U16 -> float32 weights + round-half-even + saturate;
 *            F32 -> float32; F64 -> float64 accumulation.
 *   RINT   : U8 payload sampled as int16 (uint8 image || int8 ones-mask promotes to int16): float32 weights +
 *            round-half-even. Ignored for other dtypes. */
#define OFK_ARITH_NATIVE 0
#define OFK_ARITH_RINT 1

/* rule turning the valid-weight sum S (units of 1/1024) of a warped mask into a bool (the reference's `== 1` on the
 * warped mask channel, flow_class.py:668, evaluated in the promoted dtype) */
#define OFK_RULE_STRICT 0   /* float payloads:  S == 1024 */
#define OFK_RULE_GT_HALF 1  /* int16 payloads:  S >  512  */
#define OFK_RULE_GE_HALF 2  /* uint8 payloads:  S >= 512  */

/* elementwise ops (flow_class.py:310-489) */
#define OFK_OP_ADD 0
#define OFK_OP_SUB 1
#define OFK_OP_MUL 2
#define OFK_OP_DIV 3
#define OFK_OP_POW 4

/* padding modes (flow_class.py:508-526 -> numpy.pad) */
#define OFK_PAD_CONSTANT 0
#define OFK_PAD_EDGE 1
#define OFK_PAD_SYMMETRIC 2

typedef void* ofk_stream_t; /* cudaStream_t */

const char* ofk_last_error(void);
int ofk_version(void);

/* ------------------------------------------------------------------------------------------------ hot path, device */

/* Target-referenced (backward) warp: replaces `cv2.remap(target, grid - flow, None, INTER_LINEAR)` in apply_flow
 * (utils.py:231-236) together with the mask plumbing of Flow.apply around it (flow_class.py:631-680): the mask is
 * warped in the same pass instead of being concatenated to the payload.
 *   sample position of output pixel p: p + flow_sign * flow[p]   (flow_sign = -1 for a 't' flow; +1 evaluates
 *   `flow.invert('t').apply(...)` of an 's' flow without materialising the negated field)
 *   payload      [N,Hs,Ws,C] of `dtype`;  payload_mask [N,Hs,Ws] or NULL (= all valid)
 *   flow         [N,H,W,2];               flow_mask    [N,H,W]  or NULL (= all valid), ANDed after warping
 *   top,left     position of the flow frame inside the payload frame (Flow.apply `padding`; 0,0 if Hs==H, Ws==W)
 *   cut != 0     out [N,H,W,C], out_mask [N,H,W];  cut == 0: out [N,Hs,Ws,C], out_mask [N,Hs,Ws] (flow = 0 and
 *                out_mask = 0 outside the flow frame, flow_class.py:651-660,673-678)
 *   out_mask may be NULL (no valid-area output); payload/out may be NULL with C = 0 (mask-only warp). */
int ofk_warp_t(const void* payload, int dtype, int C, int arith, const float* flow, float flow_sign,
               const uint8_t* payload_mask, const uint8_t* flow_mask, void* out, uint8_t* out_mask, int mask_rule,
               int N, int H, int W, int Hs, int Ws, int top, int left, int cut, ofk_stream_t stream);
/* ofk_warp_t_ex: flow_nonzero (int32 [N], device, e.g. from ofk_nonzero_flags(flow, NULL, 1e-3)) or NULL; frames
 * with 0 get the payload itself (its flow-frame window when cut) like apply_flow's early return for a flow that is zero
 * below the threshold (utils.py:215-216). out_mask is the same either way. Integer payloads do not need the flags:
 * identity taps reproduce them exactly; float payloads do (NaN / Inf on a zero-weight tap, -0.0). */
int ofk_warp_t_ex(const void* payload, int dtype, int C, int arith, const float* flow, float flow_sign,
                  const uint8_t* payload_mask, const uint8_t* flow_mask, const int* flow_nonzero, void* out,
                  uint8_t* out_mask, int mask_rule, int N, int H, int W, int Hs, int Ws, int top, int left, int cut,
                  ofk_stream_t stream);

/* Fused flow composition, mode 3: replaces `flow + flow.apply(self)` (ref 't', flow_class.py:1422) and
 * `self + self.invert('t').apply(flow)` (ref 's', :1418) including the zero-flow early exits (:1338-1354):
 *   ref 't': out[p] = B[p] + Q(A, p - B[p]),  out_mask[p] = Bm[p] & strict(Am taps)
 *   ref 's': out[p] = A[p] + Q(B, p + A[p]),  out_mask[p] = Am[p] & strict(Bm taps)
 * If A is zero on its valid pixels (|c| < thr when thr > 0, exact 0 otherwise) frame n of out is a copy of B (and of
 * A if B is zero), as the reference returns that operand. flags (int32 [N][2], device) receives
 * {A_nonzero, B_nonzero} per frame so the host can restore object identity; with flags == NULL the zero tests and
 * the early exits are skipped (plain composition). Am/Bm may be NULL (all valid). Mask bytes must be 0 or 1 (numpy
 * bool): the kernels AND them as words; a caller holding "non-zero = valid" bytes normalises them first (ofk_greater
 * with threshold 0 on a float copy, or host side). */
int ofk_combine3(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, int ref /* 's' or 't' */,
                 float thr, float* out, uint8_t* out_mask, int* flags, int N, int H, int W, ofk_stream_t stream);

/* Valid area of a 't'-sampling warp without payload: replaces `apply_flow(+-vecs, np.ones(shape), 't') == 1` then
 * `&= mask` in valid_target (ref 't', flow_class.py:1148-1150; flow_sign = -1) and valid_source (ref 's',
 * :1179-1183; flow_sign = +1). */
int ofk_valid_geom_t(const float* flow, float flow_sign, const uint8_t* flow_mask, uint8_t* out, int N, int H, int W,
                     ofk_stream_t stream);

/* Affine / projective field generator: replaces flow_from_matrix (utils.py:91-111). mats: N row-major 3x3 float64
 * matrices (for ref 't' the caller passes pinv(M), utils.py:343), on the host if mats_on_host != 0 (N <= 64), else on
 * the device. out[n,y,x] = sign * float32( proj(M_n [x,y,1]) - [x,y] ), float64 arithmetic in the reference's
 * rounding sequence. sign = +1 for 's', -1 for 't'. */
int ofk_from_matrix(const double* mats, int mats_on_host, float sign, float* out, int N, int H, int W,
                    ofk_stream_t stream);

/* Flow arithmetic: replaces Flow.__add__/__sub__ (flow_class.py:310-375): out = A op B (float32), and when out_mask
 * is given out_mask = Am & Bm (NULL mask = all valid). op in {OFK_OP_ADD, OFK_OP_SUB}. */
int ofk_addsub(int op, const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float* out,
               uint8_t* out_mask, int N, int H, int W, ofk_stream_t stream);

/* Per-channel scaling: replaces Flow.__mul__/__truediv__/__pow__/__neg__ (flow_class.py:377-489) for scalar and
 * 2-element multipliers: out[...,0] = A[...,0] op su, out[...,1] = A[...,1] op sv. in_f64 != 0 evaluates in float64
 * and rounds to float32 (numpy promotion for list / array operands); otherwise float32 (python-scalar operands). */
int ofk_scale(int op, const float* A, double su, double sv, int in_f64, float* out, size_t n_pixels,
              ofk_stream_t stream);

/* Array operands of the same family (also ADD / SUB of a float64 array, Flow + ndarray): M is float64 [N,H,W]
 * (m_channels = 1) or [N,H,W,2] (m_channels = 2); evaluated in float64, rounded to float32 like numpy's promotion. */
int ofk_scale_array(int op, const float* A, const double* M, int m_channels, float* out, size_t n_pixels,
                    ofk_stream_t stream);

/* Zero test gating the early exits: replaces Flow.is_zero / is_zero_flow (flow_class.py:1230-1245,
 * utils.py:527-544). flags int32 [N] (device) receives 1 where frame n has a component c with |c| >= thr
 * (thr > 0) or c != 0 (thr == 0) on a pixel whose mask is set (mask NULL = all pixels). The call zeroes flags. */
int ofk_nonzero_flags(const float* F, const uint8_t* M, float thr, int* flags, int N, int H, int W,
                      ofk_stream_t stream);

/* Finite check done by the reference in every Flow construction (flow_class.py:78-79): flag (int32, device) is set
 * to 1 if any of the n floats is NaN or +-Inf. The call zeroes flag. */
int ofk_check_finite(const float* data, size_t n, int* flag, ofk_stream_t stream);

/* Flow.pad (flow_class.py:508-526): vecs padded with mode, mask padded with 0. in [N,H,W,(2)] ->
 * out [N,H+top+bottom,W+left+right,(2)]. Either pair (vecs/out_vecs or mask/out_mask) may be NULL. */
int ofk_pad(const float* vecs, const uint8_t* mask, float* out_vecs, uint8_t* out_mask, int mode, int N, int H, int W,
            int top, int bottom, int left, int right, ofk_stream_t stream);

/* Payload dtype conversion around the float32 forward resampler (utils.py:256-258): exactly one of in_dtype /
 * out_dtype is OFK_F32, the other one of OFK_U8 / OFK_I16 / OFK_U16 / OFK_F64. From float32 to an integer type:
 * round-half-even (numpy.round) and saturate. */
int ofk_cast(const void* in, int in_dtype, void* out, int out_dtype, size_t n, ofk_stream_t stream);

/* out = a & b for 0/1 masks (the `target_mask & self.mask` of Flow.apply for 's' flows, flow_class.py:634-643). */
int ofk_mask_and(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, ofk_stream_t stream);

/* Rectangular cut of an [N,H,W] array of elem_bytes-sized items to [N,h,w] at (y0,x0): the `cut` of Flow.apply
 * (flow_class.py:663-664) and Flow.__getitem__ for contiguous windows. */
int ofk_crop(const void* in, void* out, int elem_bytes, int N, int H, int W, int y0, int x0, int h, int w,
             ofk_stream_t stream);

/* Masked extent reduction of Flow.get_padding (flow_class.py:1197-1228): out4 (float32 [N][4], device) receives
 * {min_y, max_y, min_x, max_x} of p - sign*threshold(flow)[p] over valid pixels (sign = +1 for 't', -1 for 's'). */
int ofk_extent(const float* flow, const uint8_t* mask, float sign, float thr, float* out4, int N, int H, int W,
               ofk_stream_t stream);

/* Flow.resize / resize_flow (flow_class.py:491-506, utils.py:493-524): cv2.resize(INTER_LINEAR) of vectors and float
 * mask to [N,Ho,Wo], vectors multiplied by (fx, fy) per channel, mask = round-half-even(resized mask) == 1.
 * Ho = cvRound(H*fy), Wo = cvRound(W*fx) are computed by the caller. Either pair of pointers may be NULL. */
int ofk_resize_flow(const float* vecs, const uint8_t* mask, float* out_vecs, uint8_t* out_mask, int N, int H, int W,
                    int Ho, int Wo, double fy, double fx, ofk_stream_t stream);

/* out[i] = v[i] > thr (the `> .99` mask test of combine_with mode 2 / ref 't', flow_class.py:1410). */
int ofk_greater(const float* v, float thr, uint8_t* out, size_t n, ofk_stream_t stream);

/* Flow.visualise (flow_class.py:869-951) of N frames, the one-frame call being the N = 1 case: frame n of out equals
 * Flow(flow[n], ref, mask[n]).visualise(mode, show_mask, show_mask_borders, range_max). range_max > 0: that range for every frame; range_max == 0: the reference's default per
 * frame, resolved on the device (numpy's float32 percentile(mag, 99) over all H*W magnitudes, mask ignored; if that is
 * 0 the maximum, if that is 0 too then 1); < 0 or NaN: OFK_EINVAL. mask NULL = all valid. mode 0 hsv, 1 rgb, 2 bgr.
 * out uint8 [N,H,W,3]. ws: ofk_visualise_batch_workspace(N,H,W) bytes, 4-byte aligned (256-byte aligned keeps the
 * loads of each frame's magnitudes aligned), N times a per-frame amount (0 is fine when range_max > 0). A fixed number
 * of launches whatever N (the frame index is folded into grid x, so N is not limited to 65535); H*W < 2^31. */
size_t ofk_visualise_batch_workspace(int N, int H, int W);
int ofk_visualise_batch(const float* flow, const uint8_t* mask, float thr, int mode, int show_mask,
                        int show_mask_borders, float range_max, uint8_t* out, int N, int H, int W, void* ws,
                        size_t ws_bytes, ofk_stream_t stream);

/* Flow.track (flow_class.py:755-795, utils.py:547-622) of N frames in one call: frame n of the outputs equals
 * Flow(flow[n], ref, mask[n]).track(pts_n, int_out, get_valid_status, exact), bit for bit.
 *   flow [N,H,W,2]; mask [N,H,W] or NULL (all valid), read for ref 's' status only; ref 's' or 't'.
 *   exact != 0: s_exact_mode (ref 's' float points only: Flow.track looks integer points up whatever the mode).
 *   flow_nonzero int32 [N] (device, ofk_nonzero_flags(flow, NULL, 1e-3)): frames with 0 pass their points through.
 *   pts [N,P,2] (pts_shared = 0) or [P,2] for every frame (pts_shared != 0), (row, col), of pts_dtype OFK_F32, OFK_F64,
 *     OFK_I32 or OFK_I64. Routes: ref 's' integer points look the vector up (numpy indexing: an index in [-H,-1] wraps),
 *     ref 's' float points interpolate it bilinearly in float64, or with exact locate the point in the mesh of
 *     ofk_mesh_sample on the undisplaced grid; ref 't' locates it in the mesh p - flow[p].
 *   arith OFK_F32 or OFK_F64: the type of `pts + vector` (numpy's result type; OFK_F32 only for integer points on an
 *     's' flow, i.e. numpy's int8/int16/uint8/uint16 points). out [N,P,2] of that type, or int32 with int_out != 0
 *     (round half to even).
 *   status uint8 [N,P] or NULL: valid_source at the rounded point, computed from flow and mask for ref 's' and gathered
 *     from status_plane [N,H,W] (the valid_source plane) for ref 't'.
 *   errors int32 [N] (device; the call zeroes it): bit 1 a float point on an 's' flow outside [0,H-1]x[0,W-1], bit 2 an
 *     integer point on an 's' flow outside [-H,H-1]x[-W,W-1] (both only where flow_nonzero is set), bit 4 a rounded point
 *     outside [-H,H-1]x[-W,W-1] with status. The reference raises IndexError in these cases; the call itself succeeds.
 * One kernel launch whatever N (the frame is folded into the point index). The mesh routes need H, W >= 2 and
 * H*W < 2^30. */
int ofk_track(const float* flow, const uint8_t* mask, int ref, int exact, const int* flow_nonzero, const void* pts,
              int pts_dtype, int pts_shared, int P, int arith, int int_out, void* out, const uint8_t* status_plane,
              uint8_t* status, int* errors, int N, int H, int W, ofk_stream_t stream);

/* Point trajectories through clips of flows (Sundaram, Brox & Keutzer, ECCV 2010): every point is tracked through the
 * L frames of its clip by a chain of Flow.track steps, and dropped where a step fails. flow [S*L,H,W,2] and mask
 * [S*L,H,W] (or NULL, all valid) are S clips of L frames, clip-major: frame s*L+k is the flow from frame k to frame k+1
 * of clip s. flow_nonzero int32 [S*L] (device, ofk_nonzero_flags(flow, NULL, 1e-3)). pts [S,P,2] (pts_shared = 0) or
 * [P,2] for every clip (pts_shared != 0), (row, col) in frame 0, of pts_dtype OFK_F32 or OFK_F64; a point is tracked
 * in float64. keep uint8 0/1 [S*L,H,W] or NULL (e.g. ofk_consistency of the clip's forward and backward flows).
 * One step of a live point q through frame n = s*L+k (round = half to even; "in frame" = 0 <= y <= H-1 and
 * 0 <= x <= W-1, no wrap of negative indices):
 *   ref 's' (flow on frame k's grid):
 *     1. (y, x) = round(q); lost unless in frame, valid_source of frame n at (y, x) is 1 (the per-pixel test of
 *        valid_geom with sign +1, AND the mask: Flow.track's status) and keep[n][y, x] != 0 (when given).
 *     2. q' = q where flow_nonzero[n] is 0; else ofk_track's float route, bit for bit: the float64 bilinear (lost
 *        where it raises, outside [0,H-1]x[0,W-1]), or with exact != 0 the mesh on the undisplaced grid (lost where no
 *        triangle contains q).
 *     3. lost unless round(q') is in frame.
 *   ref 't' (flow on frame k+1's grid; exact is ignored):
 *     1. lost unless round(q) is in frame.
 *     2. q' = q where flow_nonzero[n] is 0; else ofk_track's mesh p - flow[p], bit for bit (lost where no triangle
 *        contains q).
 *     3. (y', x') = round(q'); lost unless in frame, valid_target of frame n at (y', x') is 1 (valid_geom with sign -1,
 *        AND the mask) and keep[n][y', x'] != 0 (when given).
 * out float64 [S*L,P,2]: row s*L+k holds each point's position in frame k+1 of clip s, NaN from the step where the
 * point is lost to the end of its clip; alive uint8 [S*L,P] 1 / 0 likewise. One launch whatever S, L and P (one
 * thread per trajectory), none for S*P = 0; nothing is read back. S*L <= INT_MAX, frame offsets 64-bit; the mesh
 * routes need H, W >= 2 and H*W < 2^30. Every argument is checked before any device work. */
int ofk_track_clips(const float* flow, const uint8_t* mask, int ref, int exact, const int* flow_nonzero,
                    const void* pts, int pts_dtype, int pts_shared, int S, int L, int P, const uint8_t* keep,
                    double* out, uint8_t* alive, int H, int W, ofk_stream_t stream);

/* Flow.matrix (flow_class.py:797-867) of N frames: a 3x3 float64 transform per frame fitted to the point pairs of the
 * valid pixels, resolved on the device with no synchronisation.
 *   flow [N,H,W,2]; mask [N,H,W] or NULL (all valid), read when masked != 0; ref 's' (src = grid, dst = grid + flow)
 *     or 't' (src = grid - flow, dst = grid), grid = (column, row), coordinates rounded to float32.
 *   dof 4 (similarity), 6 (affine) or 8 (homography); method OFK_FIT_RANSAC or OFK_FIT_LMEDS with `hypotheses`
 *     minimal samples per frame (1 to 65536), or OFK_FIT_LMS (dof 8 only: every valid point).
 *   thr: frames whose flow is zero below thr (on valid pixels when masked) give the identity.
 *   out_mats float64 [N,3,3] (src -> dst; bottom row 0 0 1 for dof 4 and 6, H[2][2] = 1 for dof 8; all NaN for a
 *     degenerate frame); out_inliers uint8 [N,H,W] 0/1 (the inliers of the selected hypothesis, the set the refinement
 *     used) and out_counts int32 [N] (0 for zero and degenerate frames) may be NULL.
 *   ws: ofk_fit_matrix_workspace(dof, method, hypotheses, N, H, W) bytes, 8-byte aligned (0 for bad arguments).
 * Frame n of the outputs does not depend on the other frames of the batch, and repeated calls give identical outputs.
 * A fixed number of launches whatever N; N <= 65535, H*W < 2^31. */
#define OFK_FIT_LMS 0
#define OFK_FIT_RANSAC 1
#define OFK_FIT_LMEDS 2
size_t ofk_fit_matrix_workspace(int dof, int method, int hypotheses, int N, int H, int W);
int ofk_fit_matrix(const float* flow, const uint8_t* mask, int ref, int dof, int method, int hypotheses, float thr,
                   int masked, double* out_mats, uint8_t* out_inliers, int* out_counts, int N, int H, int W, void* ws,
                   size_t ws_bytes, ofk_stream_t stream);

/* Accumulation of clips of flows to their keyframe: mode-3 composition (ofk_combine3) folded over each clip, with the
 * early exits of combine_with at every step. The batch flow [S*L,H,W,2], mask [S*L,H,W] (0/1, required) is S clips
 * of L consecutive frames B_0 .. B_{L-1}, clip-major. "Zero" is the masked zero test of a whole frame at thr (as in
 * ofk_nonzero_flags); self is tested first, as in combine_with.
 *   ref 's' (left fold, frame 0 -> frame k+1 on frame 0's grid): C_0 = B_0; for k = 1 .. L-1:
 *     C_{k-1} zero -> C_k = B_k;  else B_k zero -> C_k = C_{k-1};
 *     else C_k(p) = C_{k-1}(p) + Q(B_k, p + C_{k-1}(p)), mask C_{k-1}m(p) & strict(B_k mask at the taps).
 *   ref 't' (right fold, frame j -> frame L on frame L's grid): D_{L-1} = B_{L-1}; for j = L-2 .. 0:
 *     B_j zero -> D_j = D_{j+1};  else D_{j+1} zero -> D_j = B_j;
 *     else D_j(p) = D_{j+1}(p) + Q(B_j, p - D_{j+1}(p)), mask D_{j+1}m(p) & strict(B_j mask at the taps).
 * Q is the cv2.remap sample of ofk_combine3: every frame is byte-identical to the loop of ofk_combine3 calls.
 *   cumulative != 0: out [S*L,H,W,2], out_mask [S*L,H,W], frame s*L+k = C_k ('s') or D_k ('t');
 *   cumulative == 0: out [S,H,W,2], out_mask [S,H,W], the whole-clip composite C_{L-1} ('s') or D_0 ('t').
 * flow and out 8-byte aligned; ws: ofk_accumulate_workspace(S, L) bytes, 4-byte aligned (0 for bad arguments).
 * S*L <= 65535, H and W below 32768, frame offsets 64-bit. A fixed number of launches whatever S and L: a state that
 * is zero by cancellation is found after the walk and its clip redone by one CTA (slow, exact). */
size_t ofk_accumulate_workspace(int S, int L);
int ofk_accumulate(const float* flow, const uint8_t* mask, int ref, float thr, int S, int L, int H, int W,
                   int cumulative, float* out, uint8_t* out_mask, void* ws, size_t ws_bytes, ofk_stream_t stream);

/* ofk_accumulate with the fold chosen for either ref: fold 'l' (left) or 'r' (right). The early exits depend on the
 * fold only, as in the loop of combine_with:
 *   fold 'l': A_0 = B_0; for k = 1 .. L-1: A_k = A_{k-1} (+) B_k, i.e. A_{k-1} zero -> B_k; else B_k zero -> A_{k-1};
 *     else ref 's': A_k(p) = A_{k-1}(p) + Q(B_k, p + A_{k-1}(p)), mask A_{k-1}m(p) & strict(B_k mask at the taps);
 *          ref 't': A_k(p) = B_k(p) + Q(A_{k-1}, p - B_k(p)), mask B_km(p) & strict(A_{k-1} mask at the taps).
 *   fold 'r': A_{L-1} = B_{L-1}; for j = L-2 .. 0: A_j = B_j (+) A_{j+1}, i.e. B_j zero -> A_{j+1}; else A_{j+1} zero
 *     -> B_j; else ref 's': A_j(p) = B_j(p) + Q(A_{j+1}, p + B_j(p)), mask B_jm(p) & strict(A_{j+1} mask at the taps);
 *          ref 't': A_j(p) = A_{j+1}(p) + Q(B_j, p - A_{j+1}(p)), mask A_{j+1}m(p) & strict(B_j mask at the taps).
 * ('s', 'l') and ('t', 'r') are exactly ofk_accumulate. ('t', 'l') gives the flow from frame 0 to frame k+1 on frame
 * k+1's grid (apply it to frame 0 to warp the keyframe into frame k+1); ('s', 'r') the flow from frame j to frame L
 * on frame j's grid. Outputs and cumulative as for ofk_accumulate: frame s*L+k = A_k, or one frame per clip, A_{L-1}
 * (fold 'l') or A_0 (fold 'r').
 * ws: ofk_accumulate_fold_workspace(ref, fold, S, L, H, W, cumulative) bytes (0 for bad arguments), 8-byte aligned for
 * ('t', 'l') and ('s', 'r'), 4-byte aligned otherwise. Limits as for ofk_accumulate. ('t', 'l') and ('s', 'r') sample
 * the composite of the previous step, so they run one launch per step for all S clips (L launches when cumulative,
 * max(L-1, 1) otherwise, plus 2 for the zero flags), with exact exits and no repair. */
size_t ofk_accumulate_fold_workspace(int ref, int fold, int S, int L, int H, int W, int cumulative);
int ofk_accumulate_fold(const float* flow, const uint8_t* mask, int ref, int fold, float thr, int S, int L, int H,
                        int W, int cumulative, float* out, uint8_t* out_mask, void* ws, size_t ws_bytes,
                        ofk_stream_t stream);

/* Forward-backward consistency check (Sundaram, Brox & Keutzer, ECCV 2010): occlusion masks of a pair of flows in one
 * pass. F [N,H,W,2] is the forward flow (frame 1 -> frame 2), G [N,H,W,2] the backward flow (frame 2 -> frame 1), both
 * of reference ref ('s' or 't'); the result is on F's grid. For every pixel p of frame n, in float32 with every
 * operation rounded on its own (no FMA contraction):
 *   sign = +1 ('s') or -1 ('t');  w = F[p];  (su, sv) = Q(G, p + sign * w)   (the cv2.remap sample of ofk_combine3)
 *   valid = Fm[p] & strict(Gm at the taps)                                     (the mask ofk_combine3 writes)
 *   ru = wu + su;  rv = wv + sv;  lhs = ru*ru + rv*rv
 *   rhs = alpha1 * ((wu*wu + wv*wv) + (su*su + sv*sv)) + alpha2
 *   out[p] = valid & (lhs < rhs);  out_valid[p] = valid
 * (ru, rv) and valid are the vectors and mask of ofk_combine3(F, G, 's') for ref 's' and of ofk_combine3(G, F, 't')
 * for ref 't'. There are no early exits: zero flows go through the same formula (with alpha2 = 0 a zero pair is not
 * consistent, since 0 < 0 is false). Sundaram et al. use alpha1 = 0.01, alpha2 = 0.5.
 *   Fm / Gm: uint8 0/1 masks, both given or both NULL (all valid). out, out_valid: uint8 [N,H,W]; out_valid may be
 *   NULL. F and G 8-byte aligned. alpha1, alpha2 finite and >= 0. N <= 65535, H and W below 32768, H*W below 2^30.
 * One launch whatever N: the TMA kernel of ofk_combine3 with a consistency epilogue where W % 16 == 0 and the operands
 * are 16-byte aligned, else the gather (rows) kernel of ofk_combine3 with the same epilogue; OFK_C3_WS=0 forces the
 * latter. Every argument is checked before any device work. */
int ofk_consistency(const float* F, const uint8_t* Fm, const float* G, const uint8_t* Gm, int ref, float alpha1,
                    float alpha2, uint8_t* out, uint8_t* out_valid, int N, int H, int W, ofk_stream_t stream);

/* Error metrics of N estimated flows est [N,H,W,2] against their ground truth truth [N,H,W,2] (same grid; the ref is
 * not used). Evaluated pixels: est_mask & truth_mask & region (uint8 0/1 [N,H,W] each, NULL = all valid). For every
 * pixel, with (ue, ve) = est[p], (ug, vg) = truth[p], in float32 with every operation rounded on its own (no FMA
 * contraction):
 *   du = ue - ug;  dv = ve - vg;  d2 = du*du + dv*dv;  epe = sqrt(d2)          (correctly rounded sqrt)
 *   mg = sqrt(ug*ug + vg*vg)
 *   fl = epe > 3 && epe / mg > 0.05f                                           (KITTI 2015 Fl; mg = 0 -> inf)
 *   out_k = epe > k for k = 1, 3, 5;  band = 0 if mg < 10, 1 if mg < 40, else 2  (Sintel s0-10 / s10-40 / s40+)
 *   cz = ue*vg - ve*ug;  cr = sqrt(d2 + cz*cz);  dot = (1 + ue*ug) + ve*vg
 *   ae = atan2f(cr, dot) * 57.29578f   (degrees: the angle between (ue, ve, 1) and (ug, vg, 1), Barron et al.; 0 for a
 *                                       perfect estimate)
 * Results per frame n over its evaluated pixels:
 *   counts int64 [N,8] = {evaluated, fl, out_1, out_3, out_5, band 0, band 1, band 2}
 *   sums float64 [N,5] = {epe, ae, epe over band 0, band 1, band 2}: the float32 values added in float64, per fixed
 *     block of 8192 pixels, then over the blocks in order, so a frame's rows do not depend on the batch it is in.
 *   epe float32 [N,H,W] or NULL: the EPE of every pixel, evaluated or not.
 * Inputs whose squares overflow give inf (and NaN where inf meets inf) as float32 arithmetic does.
 * est and truth 8-byte aligned (16 for vector loads), ws: ofk_evaluate_workspace(N, H, W) bytes, 8-byte aligned (0 for
 * bad arguments). N <= 65535, H*W < 2^31. Every argument is checked before any device work. Two launches whatever N
 * (per-block partials, then one fixed-order pass per frame), none for N = 0. */
size_t ofk_evaluate_workspace(int N, int H, int W);
int ofk_evaluate(const float* est, const uint8_t* est_mask, const float* truth, const uint8_t* truth_mask,
                 const uint8_t* region, float* epe, long long* counts, double* sums, int N, int H, int W, void* ws,
                 size_t ws_bytes, ofk_stream_t stream);

/* points_inside_area (utils.py:283-295): pts float64 [n][2] (row, col) rounded half-even like numpy.round. */
int ofk_points_inside_area(const double* pts, size_t n, int H, int W, uint8_t* out, ofk_stream_t stream);

/* Dataset decoders (the data formats either side of the path, utils.py:426-490). ofk_decode_kitti: bgr is the uint16
 * [n_pixels][3] image exactly as cv2.imread(path, IMREAD_UNCHANGED) returns it (load_kitti, utils.py:426-445);
 * vecs[i] = ((R - 2^15) / 64, (G - 2^15) / 64) in float32 (exact), mask[i] = B != 0 (Flow.from_kitti with load_valid;
 * mask may be NULL). ofk_decode_sintel_mask: the invalid-pixel image of load_sintel_mask (utils.py:474-490),
 * mask = (invalid == 0). A Sintel .flo payload is float32 (u, v) already and is uploaded as is. */
int ofk_decode_kitti(const uint16_t* bgr, float* vecs, uint8_t* mask, size_t n_pixels, ofk_stream_t stream);
int ofk_decode_sintel_mask(const uint8_t* invalid, uint8_t* mask, size_t n_pixels, ofk_stream_t stream);

/* ------------------------------------------------------------------------------- source-referenced path, device */

/* Source-referenced (forward) resampling: replaces `griddata(grid + flow, payload, grid, 'linear')` + nan_to_num in
 * apply_flow (utils.py:237-258): the Delaunay triangulation of the displaced pixel positions p + flow_sign * flow[p]
 * with barycentric interpolation (float64 geometry) and 0 outside the convex hull. Cells of the displaced grid with
 * four valid corners are rasterised directly (each split along its Delaunay diagonal); everything else is covered by
 * the Delaunay triangles of the boundary points, exactly as Qhull bridges them: the pockets between the displaced frame
 * border and its convex hull (frames without removed points) and the small faces left by removed points are
 * triangulated explicitly and rasterised with the same fill rule, what remains (large or border-touching faces) is
 * located per pixel in the triangulation of the boundary points. A frame whose point_mask removes nothing is treated
 * like one without a point mask (tested per frame on the device).
 *   payload       float32 [N,H,W,C]; payload_mask [N,H,W] (or NULL = all valid) is resampled with it and turned into
 *                 out_mask by mask_rule: OFK_RULE_STRICT (float payloads: interpolated mask == 1 after the float32
 *                 cast) or OFK_RULE_GT_HALF (integer payloads: numpy.round(interpolated mask) == 1)
 *   point_mask    [N,H,W] or NULL: `consider_mask`, the points with 0 are removed before triangulating (utils.py:249-251)
 *   mask bytes    must be 0 or 1
 *   ws            device workspace of ofk_forward_s_workspace(N,H,W) bytes; payload/out may be NULL with C = 0
 * Folding fields (a displaced cell with a non-positive triangle anywhere in the frame): such a frame is triangulated
 * as a whole -- every kept point is a vertex of the Delaunay triangulation griddata builds, and every pixel is located
 * in it -- so the result is griddata's, at a far higher cost than a frame that does not fold.
 * ofk_forward_s_ex: flow_nonzero (int32 [N], device, e.g. from ofk_nonzero_flags(flow, NULL, 1e-3)) or NULL; frames
 * with 0 are passed through (out = payload, out_mask = payload_mask) like apply_flow's early return for a flow that is
 * zero below the threshold (utils.py:215-216).
 * Asynchronous on `stream` like every ofk_* call; internally the part that does not depend on the cell rasteriser runs
 * on a library-owned side stream per device, forked from and joined back into `stream` with events inside the call. */
size_t ofk_forward_s_workspace(int N, int H, int W);
int ofk_forward_s(const float* payload, int C, const float* flow, float flow_sign, const uint8_t* payload_mask,
                  const uint8_t* point_mask, float* out, uint8_t* out_mask, int mask_rule, int N, int H, int W,
                  void* ws, size_t ws_bytes, ofk_stream_t stream);
int ofk_forward_s_ex(const float* payload, int C, const float* flow, float flow_sign, const uint8_t* payload_mask,
                     const uint8_t* point_mask, const int* flow_nonzero, float* out, uint8_t* out_mask, int mask_rule,
                     int N, int H, int W, void* ws, size_t ws_bytes, ofk_stream_t stream);

/* Test hook: switches passes of ofk_forward_s off for subsequent calls of this process (0 = production): 4 the pocket
 * pass, 8 the small-face pass, 16 the tracing of a mask's outer boundary. What they would have produced is then located
 * per pixel -- the same triangulation by another route (tests assert equal results). */
int ofk_forward_s_set_disable(int passes);

/* Test hook: cells of the displaced grid whose in-circle determinant is within +-tol take the OTHER diagonal in
 * subsequent ofk_forward_s calls of this process (0 = production behaviour). Similarity transforms leave the four
 * corners of a cell co-circular to within rounding; Qhull's diagonal there is arbitrary, and the parity tests compare
 * the reference against both answers. */
int ofk_forward_s_set_flip_tol(double tol);

/* Scattered-to-scattered barycentric interpolation on the displaced-grid mesh: replaces the direct
 * `griddata(grid - A, A||mask, grid - B, 'linear', fill_value=0)` of combine_with mode 2 / ref 't'
 * (flow_class.py:1398-1410) and the griddata calls of track_pts (utils.py:603,614).
 *   mesh vertices: p + mesh_sign * mesh_flow[p] carrying payload[p] (float32, C channels) and payload_mask[p]
 *   queries: either one per pixel at p + query_sign * query_flow[p] (Q = H*W), or Q explicit float64 (row, col)
 *   points per frame (query_pts [N,Q,2]); exactly one of the two is non-NULL.
 *   pos_f32 != 0: coordinates are rounded to float32 before use, as the reference's in-place float32 adds do.
 *   out [N,Q,C] float32 (0 outside the mesh), out_maskval [N,Q] float32 interpolated mask (may be NULL),
 *   found [N,Q] uint8: 1 where a containing triangle exists (griddata returns NaN elsewhere; may be NULL). */
int ofk_mesh_sample(const float* mesh_flow, float mesh_sign, int pos_f32, const float* payload, int C,
                    const uint8_t* payload_mask, const float* query_flow, float query_sign, const double* query_pts,
                    int Q, float* out, float* out_maskval, uint8_t* found, int N, int H, int W, ofk_stream_t stream);

/* Flow composition, modes 1 and 2 (flow_class.py:1357-1410), frame-wise on a batch: the chains of forward / backward
 * warps, additions and mask-ANDs the reference writes as Flow methods, run on the device behind one call.
 *   mode 1: flow_1 such that flow_1 (+) A = B;   mode 2: flow_2 such that A (+) flow_2 = B;   ref 's' or 't' (both
 *   operands and the result). Am / Bm may be NULL (all valid); mask bytes must be 0 or 1.
 * The zero-flow tests INSIDE the chains (switch_ref relabels an exactly-zero flow, apply_flow passes its target through
 * for a flow below the threshold) are evaluated per frame on the device. The early exits of combine_with itself
 * (:1338-1354: A zero -> B, B zero -> A.invert()) return operand objects and stay with the caller
 * (ofk_nonzero_flags). ws: device workspace of ofk_combine12_workspace(mode, ref, N, H, W) bytes.
 * ofk_combine2_t is mode 2 / ref 't' alone (one launch, no workspace): B - resample(A, grid - A -> grid - B). */
size_t ofk_combine12_workspace(int mode, int ref, int N, int H, int W);
int ofk_combine12(int mode, int ref, const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float* out,
                  uint8_t* out_mask, int N, int H, int W, void* ws, size_t ws_bytes, ofk_stream_t stream);
int ofk_combine2_t(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float* out, uint8_t* out_mask,
                   int N, int H, int W, ofk_stream_t stream);

/* ------------------------------------------------------------------------------------------------ host-buffer API */

/* Same operations on HOST buffers (what `apply_flow(flow, img, 't')` / `Flow.apply(..., return_valid_area=True)` and
 * `combine_flows(a, b, 3, ref)` / `Flow.combine_with` look like from numpy): frames are streamed through an internal
 * ring of pinned staging + device buffers on `device`, copies overlapped with kernels. Synchronous. */
int ofh_warp_t(const void* payload, int dtype, int C, int arith, const float* flow, float flow_sign,
               const uint8_t* payload_mask, const uint8_t* flow_mask, void* out, uint8_t* out_mask, int mask_rule,
               int N, int H, int W, int device);
int ofh_combine3(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, int ref, float thr, float* out,
                 uint8_t* out_mask, int* flags, int N, int H, int W, int device);
/* `A.apply(image, return_valid_area)` + `A.combine_with(B, 3)` of a batch in ONE pass of the ring: A and its mask are
 * uploaded once and feed both kernels (the two calls above upload them twice). A is the warping flow (ref 't': sample
 * at p - A[p]; ref 's' is accepted for the composition, the image warp then samples at p + A[p], i.e.
 * `A.invert('t').apply(image)`). out_valid may be NULL (no valid area); flags as in ofk_combine3 (may be NULL). */
int ofh_apply_combine3(const void* image, int dtype, int C, int arith, int mask_rule, const float* A, const uint8_t* Am,
                       const float* B, const uint8_t* Bm, int ref, float thr, void* out_image, uint8_t* out_valid,
                       float* out, uint8_t* out_mask, int* flags, int N, int H, int W, int device);
/* ofk_visualise_batch on host buffers (flow [N,H,W,2], mask [N,H,W] or NULL, out uint8 [N,H,W,3]) through the ring;
 * synchronous. */
int ofh_visualise(const float* flow, const uint8_t* mask, float thr, int mode, int show_mask, int show_mask_borders,
                  float range_max, uint8_t* out, int N, int H, int W, int device);
/* ofk_evaluate on host buffers through the ring; synchronous. Only the per-frame rows (104 bytes per frame) and, if
 * epe is not NULL, the EPE map come back. */
int ofh_evaluate(const float* est, const uint8_t* est_mask, const float* truth, const uint8_t* truth_mask,
                 const uint8_t* region, float* epe, long long* counts, double* sums, int N, int H, int W, int device);
/* All ofh_* calls leave the caller's current CUDA device unchanged. */
/* release the internal ring (also done at process exit) */
int ofh_release(void);

/* ------------------------------------------------------------------------------------------------------- runtime */
int ofk_rt_device_count(int* count);
int ofk_rt_set_device(int device);
int ofk_rt_get_device(int* device);
int ofk_rt_device_info(int device, int* sm_count, int* cc_major, int* cc_minor, size_t* l2_bytes, size_t* total_mem);
int ofk_rt_malloc(void** dptr, size_t bytes, ofk_stream_t stream); /* stream-ordered pool allocation, current device */
int ofk_rt_free(void* dptr, ofk_stream_t stream);
int ofk_rt_host_alloc(void** hptr, size_t bytes);          /* pinned */
int ofk_rt_host_free(void* hptr);
int ofk_rt_host_register(void* hptr, size_t bytes);        /* pin an existing numpy buffer */
int ofk_rt_host_unregister(void* hptr);
/* Host <-> device copies, stream-ordered. Pinned / registered host memory: plain asynchronous copies. Pageable host
 * memory (ordinary numpy arrays) of 4 MiB and more: worker threads stage 2 MiB pieces through pinned buffers so the copy
 * runs near PCIe rate instead of the driver's single-threaded staging; h2d returns once the source has been read,
 * d2h once the destination is complete (as cudaMemcpyAsync behaves for pageable memory). OFK_STAGED_COPIES=0 disables. */
int ofk_rt_memcpy_h2d(void* dst, const void* src, size_t bytes, ofk_stream_t stream);
int ofk_rt_memcpy_d2h(void* dst, const void* src, size_t bytes, ofk_stream_t stream);
int ofk_rt_memcpy_d2d(void* dst, const void* src, size_t bytes, ofk_stream_t stream);
int ofk_rt_memset(void* dst, int value, size_t bytes, ofk_stream_t stream);
int ofk_rt_stream_create(ofk_stream_t* stream);
int ofk_rt_stream_destroy(ofk_stream_t stream);
int ofk_rt_stream_sync(ofk_stream_t stream);
int ofk_rt_device_sync(void);
int ofk_rt_event_create(void** event);
int ofk_rt_event_destroy(void* event);
int ofk_rt_event_record(void* event, ofk_stream_t stream);
int ofk_rt_stream_wait_event(ofk_stream_t stream, void* event);   /* work queued later on stream waits for event */
int ofk_rt_event_sync(void* event);
int ofk_rt_event_elapsed_ms(void* start, void* stop, float* ms);
/* number of kernel launches issued by this library in this process (bench.py's gpu_launches) */
unsigned long long ofk_rt_launch_count(void);
/* how often each implementation of the two headline operations ran (tests assert that eligible shapes take the TMA
 * kernels): which = 0 ofk_combine3 / TMA kernel, 1 ofk_combine3 / gather kernels, 2 ofk_warp_t / TMA kernels,
 * 3 ofk_warp_t / gather kernels. which = 4 / 5: inside the TMA kernels of ofk_combine3 / ofk_warp_t, how many
 * (warp, tile) pairs fetched taps from global memory because the tile's box did not cover them (discontinuous or noisy
 * flows); read synchronously from the current device. Counter 4 also counts ofk_consistency's TMA kernel, which is the
 * same kernel. which = 6..9: ofk_forward_s, pixels outside the regular mesh
 * since process start: 6 located in a bridging / pocket triangle, 7 found outside the hull by the search, 8 searches
 * that did not terminate (treated as outside; expected 0), 9 rejected by the per-frame hull polygon, 10 pixels handed
 * to the warp-cooperative pocket pass, 11 its work items. which = 12 / 13: ofk_consistency calls that ran the TMA
 * kernel / the gather (rows) kernel. */
unsigned long long ofk_rt_path_count(int which);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* OFLIB_B200_H */
