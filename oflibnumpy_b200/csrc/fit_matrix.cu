// Transformation matrices fitted to N flows at once, ofk_fit_matrix: the batched, device-resolved form of Flow.matrix
// (flow_class.py:797-867: cv2.estimateAffinePartial2D / estimateAffine2D / findHomography on the point pairs of every
// valid pixel). Every stage is a fixed number of launches over all frames; blocks are numbered frame-major on grid x.
//
//   zero flags     : ofk_nonzero_flags (with the mask when masked); a zero frame gives the identity.
//   valid list     : masked -> the valid pixel indices of each frame in raster order (count / per-frame scan / scatter).
//   hypotheses     : one thread per (frame, k): a minimal sample of 2 / 3 / 4 list entries drawn with splitmix64
//                    (the key holds k and the draw counter, never the frame: a frame gives the same result in any
//                    batch), degeneracy tests, closed-form / Gaussian-elimination minimal solvers in float64 with
//                    explicit _rn intrinsics (no contraction) so that a numpy restatement reproduces them bit for bit.
//   scoring        : blocks of (frame, group of hypotheses, chunk of pixels); each point is formed once and scored
//                    against the group. RANSAC counts float32 residuals <= 9; LMedS finds the residual of rank M/2 of
//                    every (frame, hypothesis) segment by the radix selection of radix_select.cuh, recomputing the
//                    residuals in each pass. Integer atomics only.
//   selection      : best score per frame, ties to the lowest k; the inlier threshold.
//   refinement     : fixed-size per-block float64 partials, summed per frame in a fixed order, on the inliers of the
//                    selected hypothesis (lms: every valid point), in coordinates centred on the frame centre.
//                    dof 4 / 6: normal equations of the linear least-squares problem. dof 8: normalised DLT (centroid,
//                    mean absolute deviation, 9x9 L^T L, smallest eigenvector by one-thread Jacobi), then 10
//                    Levenberg-Marquardt steps on the forward reprojection error, one reduction launch each, the step
//                    accepted or rejected on the device.
#include <stddef.h>

#include <algorithm>
#include <cfloat>

#include "radix_select.cuh"

namespace ofk {
namespace fit {

#define DADD __dadd_rn
#define DSUB __dsub_rn
#define DMUL __dmul_rn
#define DDIV __ddiv_rn

constexpr int kChunk = 8192;            // pixels per block of the list and refinement kernels (fixed: the partial
                                        // sums of a frame do not depend on the batch)
constexpr int kCountG = 8, kCountChunk = 4096;    // RANSAC scoring: hypotheses x pixels per block
constexpr int kHistG = 2, kHistChunk = 16384;     // LMedS histogram passes
constexpr int kMaxSums = 45;
constexpr int kTries = 8;               // draws per sample point before the hypothesis counts as degenerate
constexpr int kLmIters = 10;            // findHomography's LM iteration limit
constexpr unsigned long long kSeed = 0x6f666c69625f6669ull;

enum Status { kZero = 0, kFit = 1, kDegenerate = 2 };
enum Stage { kSim = 0, kAff = 1, kCen = 2, kMad = 3, kLtl = 4, kLm = 5 };
__host__ __device__ constexpr int stage_sums(int st) {
    return st == kSim ? 8 : st == kAff ? 12 : st == kCen ? 5 : st == kMad ? 4 : 45;
}

struct Frame {
    int status, M, best, count;
    float thr2;
    int pad;
    double model[9];          // the selected hypothesis, pixel coordinates, model[8] = 1
    double cen[4], scl[4];    // dof 8 DLT: centroids and scales of src (x, y) and dst (x, y), centred coordinates
    double h[8], cand[8];     // dof 8 LM: accepted and candidate homography in centred coordinates (h[8] = 1)
    double err, lambda;
    double jtj[36], jte[8];   // at h
};

struct Pt {
    double sx, sy, dx, dy;
};

// The point pair of pixel p (x = column, y = row): ref 's' src = grid, dst = fl32(grid + flow); ref 't' dst = grid,
// src = fl32(grid - flow).
__device__ __forceinline__ Pt make_point(const float2* f, size_t p, int W, int ref) {
    const int y = (int)(p / (size_t)W), x = (int)(p - (size_t)y * W);
    const float2 v = __ldg(f + p);
    const float fx = (float)x, fy = (float)y;
    if (ref == 's') return {fx, fy, __fadd_rn(fx, v.x), __fadd_rn(fy, v.y)};
    return {__fsub_rn(fx, v.x), __fsub_rn(fy, v.y), fx, fy};
}

// Squared reprojection distance |M src - dst|^2, dof 8 projected through w (cv2's computeError), rounded to float32;
// NaN counts as +inf.
template <bool HOMOG>
__device__ __forceinline__ float residual(const double* m, const Pt& q) {
    double px = DADD(DADD(DMUL(m[0], q.sx), DMUL(m[1], q.sy)), m[2]);
    double py = DADD(DADD(DMUL(m[3], q.sx), DMUL(m[4], q.sy)), m[5]);
    if (HOMOG) {
        const double iw = DDIV(1.0, DADD(DADD(DMUL(m[6], q.sx), DMUL(m[7], q.sy)), 1.0));
        px = DMUL(px, iw);
        py = DMUL(py, iw);
    }
    const double ex = DSUB(px, q.dx), ey = DSUB(py, q.dy);
    const float r = __double2float_rn(DADD(DMUL(ex, ex), DMUL(ey, ey)));
    return r != r ? __int_as_float(0x7f800000) : r;
}

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long seed, unsigned k, unsigned c) {
    unsigned long long z = seed + (((unsigned long long)k << 32) | c) * 0x9e3779b97f4a7c15ull;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

// Gaussian elimination with partial pivoting (first maximum on ties); false if a pivot is 0 or the solution is not
// finite. A and b are overwritten.
template <int NN>
__device__ bool gauss_solve(double (&A)[NN][NN], double (&b)[NN], double (&x)[NN]) {
    for (int c = 0; c < NN; ++c) {
        int p = c;
        double best = fabs(A[c][c]);
        for (int r = c + 1; r < NN; ++r)
            if (fabs(A[r][c]) > best) {
                best = fabs(A[r][c]);
                p = r;
            }
        if (!(best != 0.0)) return false;
        if (p != c) {
            for (int j = 0; j < NN; ++j) {
                const double t = A[c][j];
                A[c][j] = A[p][j];
                A[p][j] = t;
            }
            const double t = b[c];
            b[c] = b[p];
            b[p] = t;
        }
        for (int r = c + 1; r < NN; ++r) {
            const double f = DDIV(A[r][c], A[c][c]);
            for (int j = c + 1; j < NN; ++j) A[r][j] = DSUB(A[r][j], DMUL(f, A[c][j]));
            b[r] = DSUB(b[r], DMUL(f, b[c]));
        }
    }
    bool ok = true;
    for (int i = NN - 1; i >= 0; --i) {
        double s = b[i];
        for (int j = i + 1; j < NN; ++j) s = DSUB(s, DMUL(A[i][j], x[j]));
        x[i] = DDIV(s, A[i][i]);
        ok = ok && isfinite(x[i]);
    }
    return ok;
}

// Points a, b, c collinear or coincident, seen from c (cv2's haveCollinearPoints test).
__device__ __forceinline__ bool collinear(const double* x, const double* y, int a, int b, int c) {
    const double dx1 = DSUB(x[a], x[c]), dy1 = DSUB(y[a], y[c]), dx2 = DSUB(x[b], x[c]), dy2 = DSUB(y[b], y[c]);
    const double cr = DSUB(DMUL(dx2, dy1), DMUL(dy2, dx1));
    const double s = DADD(DADD(DADD(fabs(dx1), fabs(dy1)), fabs(dx2)), fabs(dy2));
    return fabs(cr) <= DMUL((double)FLT_EPSILON, s);
}

__device__ __forceinline__ double orient(const double* x, const double* y, int a, int b, int c) {
    return DSUB(DMUL(DSUB(x[b], x[a]), DSUB(y[c], y[a])), DMUL(DSUB(y[b], y[a]), DSUB(x[c], x[a])));
}

// ------------------------------------------------------------------------------------------------ valid-pixel list
__global__ void __launch_bounds__(256) list_count_kernel(const uint8_t* __restrict__ mask, int* __restrict__ cnt,
                                                         size_t hw, int bpf) {
    const size_t n = blockIdx.x / bpf, b = blockIdx.x - n * bpf;
    int c = 0;
    for (int j = 0; j < kChunk / 256; ++j) {
        const size_t p = b * kChunk + j * 256 + threadIdx.x;
        c += __syncthreads_count(p < hw && mask[n * hw + p]);
    }
    if (threadIdx.x == 0) cnt[blockIdx.x] = c;
}

// One thread per frame: per-block offsets of the list (in place), M, the frame's status and initial state.
__global__ void frames_kernel(const int* __restrict__ nonzero, int* __restrict__ cnt, Frame* __restrict__ fr, int N,
                              int hw, int bpf, int use_list, int s) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    int M = hw;
    if (use_list) {
        M = 0;
        for (int b = 0; b < bpf; ++b) {
            const int c = cnt[(size_t)n * bpf + b];
            cnt[(size_t)n * bpf + b] = M;
            M += c;
        }
    }
    Frame& F = fr[n];
    F.status = nonzero[n] == 0 ? kZero : (M < s ? kDegenerate : kFit);
    F.M = M;
    F.best = -1;
    F.count = 0;
    F.thr2 = __int_as_float(0x7f800000);
    F.lambda = 1e-3;
}

__global__ void __launch_bounds__(256) list_scatter_kernel(const uint8_t* __restrict__ mask,
                                                           const int* __restrict__ off, int* __restrict__ list,
                                                           size_t hw, int bpf) {
    __shared__ int wc[8];
    const size_t n = blockIdx.x / bpf, b = blockIdx.x - n * bpf;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int run = off[blockIdx.x];
    for (int j = 0; j < kChunk / 256; ++j) {
        const size_t p = b * kChunk + j * 256 + threadIdx.x;
        const bool v = p < hw && mask[n * hw + p];
        const unsigned bal = __ballot_sync(0xffffffffu, v);
        if (lane == 0) wc[wid] = __popc(bal);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < 8; ++w) {
            before += w < wid ? wc[w] : 0;
            total += wc[w];
        }
        if (v) list[n * hw + run + before + __popc(bal & ((1u << lane) - 1u))] = (int)p;
        run += total;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ hypotheses
template <int DOF>
__global__ void __launch_bounds__(128) hypotheses_kernel(const float2* __restrict__ flow, const int* __restrict__ list,
                                                         const Frame* __restrict__ fr, double* __restrict__ models,
                                                         int* __restrict__ ok, int K, size_t total, int hw, int W,
                                                         int ref) {
    constexpr int S = DOF / 2;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const size_t n = t / K;
    const unsigned k = (unsigned)(t - n * K);
    ok[t] = 0;
    if (fr[n].status != kFit) return;
    const unsigned long long M = (unsigned long long)fr[n].M;
    unsigned idx[S];
    unsigned c = 0;
    for (int j = 0; j < S; ++j) {
        int tr = 0;
        for (; tr < kTries; ++tr) {
            const unsigned id = (unsigned)(((splitmix64(kSeed, k, c++) >> 32) * M) >> 32);
            bool rep = false;
            for (int i = 0; i < j; ++i) rep = rep || idx[i] == id;
            if (!rep) {
                idx[j] = id;
                break;
            }
        }
        if (tr == kTries) return;
    }
    double sx[S], sy[S], dx[S], dy[S];
    for (int j = 0; j < S; ++j) {
        const size_t p = list ? (size_t)list[n * hw + idx[j]] : idx[j];
        const Pt q = make_point(flow + n * hw, p, W, ref);
        sx[j] = q.sx, sy[j] = q.sy, dx[j] = q.dx, dy[j] = q.dy;
    }
    double m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 1};
    if (DOF == 4) {
        const double ux = DSUB(sx[1], sx[0]), uy = DSUB(sy[1], sy[0]), vx = DSUB(dx[1], dx[0]), vy = DSUB(dy[1], dy[0]);
        const double den = DADD(DMUL(ux, ux), DMUL(uy, uy));
        if (den == 0.0 || (vx == 0.0 && vy == 0.0)) return;
        const double a = DDIV(DADD(DMUL(vx, ux), DMUL(vy, uy)), den);
        const double b = DDIV(DSUB(DMUL(vy, ux), DMUL(vx, uy)), den);
        m[0] = a, m[1] = -b, m[3] = b, m[4] = a;
        m[2] = DSUB(dx[0], DSUB(DMUL(a, sx[0]), DMUL(b, sy[0])));
        m[5] = DSUB(dy[0], DADD(DMUL(b, sx[0]), DMUL(a, sy[0])));
        if (!(isfinite(m[0]) && isfinite(m[1]) && isfinite(m[2]) && isfinite(m[5]))) return;
    } else if (DOF == 6) {
        if (collinear(sx, sy, 0, 1, 2) || collinear(dx, dy, 0, 1, 2)) return;
        for (int r = 0; r < 2; ++r) {
            double A[3][3], b[3], x[3];
            for (int i = 0; i < 3; ++i) {
                A[i][0] = sx[i], A[i][1] = sy[i], A[i][2] = 1.0;
                b[i] = r == 0 ? dx[i] : dy[i];
            }
            if (!gauss_solve<3>(A, b, x)) return;
            m[3 * r] = x[0], m[3 * r + 1] = x[1], m[3 * r + 2] = x[2];
        }
    } else {
        const int tri[4][3] = {{0, 1, 2}, {1, 2, 3}, {0, 2, 3}, {0, 1, 3}};
        int negative = 0;
        for (int i = 0; i < 4; ++i) {
            const int a = tri[i][0], b = tri[i][1], cc = tri[i][2];
            if (collinear(sx, sy, a, b, cc) || collinear(dx, dy, a, b, cc)) return;
            negative += DMUL(orient(sx, sy, a, b, cc), orient(dx, dy, a, b, cc)) < 0.0;
        }
        if (negative != 0 && negative != 4) return;
        double A[8][8], b[8], x[8];
        for (int i = 0; i < 4; ++i) {
            double* r0 = A[2 * i];
            double* r1 = A[2 * i + 1];
            r0[0] = sx[i], r0[1] = sy[i], r0[2] = 1.0, r0[3] = 0.0, r0[4] = 0.0, r0[5] = 0.0;
            r0[6] = -DMUL(sx[i], dx[i]), r0[7] = -DMUL(sy[i], dx[i]);
            r1[0] = 0.0, r1[1] = 0.0, r1[2] = 0.0, r1[3] = sx[i], r1[4] = sy[i], r1[5] = 1.0;
            r1[6] = -DMUL(sx[i], dy[i]), r1[7] = -DMUL(sy[i], dy[i]);
            b[2 * i] = dx[i], b[2 * i + 1] = dy[i];
        }
        if (!gauss_solve<8>(A, b, x)) return;
        for (int i = 0; i < 8; ++i) m[i] = x[i];
    }
    for (int i = 0; i < 9; ++i) models[t * 9 + i] = m[i];
    ok[t] = 1;
}

// ------------------------------------------------------------------------------------------------ scoring
// PASS < 0: RANSAC inlier counts; PASS 0..2: LMedS histogram pass. Block = (frame, group of G hypotheses, chunk).
template <bool HOMOG, int PASS>
__global__ void __launch_bounds__(256) score_kernel(const float2* __restrict__ flow, const uint8_t* __restrict__ mask,
                                                    const Frame* __restrict__ fr, const double* __restrict__ models,
                                                    const int* __restrict__ ok, unsigned* __restrict__ counts,
                                                    const uint2* __restrict__ sel, unsigned* __restrict__ hist, int K,
                                                    int hw, int W, int ref, int groups, int chunks) {
    constexpr int G = PASS < 0 ? kCountG : kHistG, kPts = PASS < 0 ? kCountChunk : kHistChunk;
    constexpr int kBins = PASS < 0 ? 1 : pass_bins(PASS), kShift = PASS < 0 ? 0 : pass_shift(PASS);
    constexpr unsigned kHiMask = PASS <= 0 ? 0u : ~0u << (kShift + 10);
    __shared__ double sm[G][9];
    __shared__ int sok[G];
    __shared__ unsigned spre[G];
    __shared__ unsigned sh[G * kBins];
    const size_t n = blockIdx.x / ((size_t)groups * chunks);
    const int r = (int)(blockIdx.x - n * groups * chunks), g0 = (r / chunks) * G, c = r % chunks;
    if (fr[n].status != kFit) return;
    const size_t seg0 = n * K + g0;
    if (threadIdx.x < G * 9) {
        const int g = threadIdx.x / 9;
        sm[g][threadIdx.x % 9] = g0 + g < K ? models[(seg0 + g) * 9 + threadIdx.x % 9] : 0.0;
    }
    if (threadIdx.x < G) {
        const int g = threadIdx.x;
        sok[g] = g0 + g < K && ok[seg0 + g];
        spre[g] = (PASS > 0 && sok[g]) ? sel[seg0 + g].x : 0u;
    }
    for (int k = threadIdx.x; k < G * kBins; k += blockDim.x) sh[k] = 0;
    __syncthreads();
    const float2* f = flow + n * hw;
    const uint8_t* mk = mask ? mask + n * hw : nullptr;
    const int start = c * kPts, end = min(start + kPts, hw);
    int cnt[G];
#pragma unroll
    for (int g = 0; g < G; ++g) cnt[g] = 0;
    for (int base = start; base < end; base += 256) {
        const int p = base + threadIdx.x;
        const bool in = p < end && (mk == nullptr || mk[p]);
        const Pt q = make_point(f, in ? p : start, W, ref);
#pragma unroll
        for (int g = 0; g < G; ++g) {
            if (!sok[g]) continue;                                   // uniform over the block
            const float e = residual<HOMOG>(sm[g], q);
            if (PASS < 0) {
                cnt[g] += in && e <= 9.0f;
            } else {
                const unsigned bits = __float_as_uint(e);
                hist_add(sh + g * kBins, (bits >> kShift) & (kBins - 1), in && (bits & kHiMask) == spre[g]);
            }
        }
    }
    if (PASS < 0) {
#pragma unroll
        for (int g = 0; g < G; ++g) {
            const unsigned v = __reduce_add_sync(0xffffffffu, (unsigned)cnt[g]);
            if ((threadIdx.x & 31) == 0 && v) atomicAdd(sh + g, v);
        }
        __syncthreads();
        if (threadIdx.x < G && sok[threadIdx.x] && sh[threadIdx.x]) atomicAdd(counts + seg0 + threadIdx.x, sh[threadIdx.x]);
    } else {
        __syncthreads();
        for (int g = 0; g < G; ++g)
            if (sok[g]) flush_hist(sh + g * kBins, hist + (seg0 + g) * kBins0, kBins);
    }
}

// One warp per (frame, hypothesis) segment: the bin of this pass holding rank M/2 (or the rank left from the previous
// pass); the histogram is zeroed for the next pass.
template <int PASS>
__global__ void __launch_bounds__(256) pick_kernel(const Frame* __restrict__ fr, const int* __restrict__ ok,
                                                   uint2* __restrict__ sel, unsigned* __restrict__ hist, int K,
                                                   size_t segs) {
    constexpr int kBins = pass_bins(PASS), kShift = pass_shift(PASS), kPer = kBins / 32;
    const size_t seg = (size_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (seg >= segs || fr[seg / K].status != kFit || !ok[seg]) return;
    unsigned* h = hist + seg * kBins0 + lane * kPer;
    const unsigned rank = PASS == 0 ? (unsigned)(fr[seg / K].M / 2) : sel[seg].y;
    unsigned local = 0;
    for (int k = 0; k < kPer; ++k) local += h[k];
    unsigned incl = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const unsigned excl = incl - local;
    if (excl <= rank && rank < incl) {
        unsigned r = rank - excl;
        int bin = lane * kPer + kPer - 1;
        for (int k = 0; k < kPer; ++k) {
            if (r < h[k]) {
                bin = lane * kPer + k;
                break;
            }
            r -= h[k];
        }
        sel[seg] = make_uint2((PASS == 0 ? 0u : sel[seg].x) | ((unsigned)bin << kShift), r);
    }
    for (int k = 0; k < kPer; ++k) h[k] = 0;
}

// One block per frame: the best hypothesis (RANSAC: most inliers, LMedS: smallest median; ties to the lowest k) and
// the inlier threshold; no valid hypothesis -> degenerate.
__global__ void __launch_bounds__(256) select_kernel(Frame* __restrict__ fr, const double* __restrict__ models,
                                                     const int* __restrict__ ok, const unsigned* __restrict__ counts,
                                                     const uint2* __restrict__ sel, int K, int lmeds, int s) {
    __shared__ unsigned long long wmin[8];
    const size_t n = blockIdx.x;
    Frame& F = fr[n];
    if (F.status != kFit) return;
    unsigned long long key = ~0ull;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        const size_t seg = n * K + k;
        if (!ok[seg]) continue;
        const unsigned score = lmeds ? sel[seg].x : 0xffffffffu - counts[seg];
        key = min(key, ((unsigned long long)score << 32) | (unsigned)k);
    }
    for (int o = 16; o > 0; o >>= 1) key = min(key, __shfl_down_sync(0xffffffffu, key, o));
    if ((threadIdx.x & 31) == 0) wmin[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x != 0) return;
    for (int w = 1; w < 8; ++w) key = min(key, wmin[w]);
    if (key == ~0ull) {
        F.status = kDegenerate;
        return;
    }
    const int k = (int)(key & 0xffffffffu);
    F.best = k;
    for (int i = 0; i < 9; ++i) F.model[i] = models[(n * K + k) * 9 + i];
    if (!lmeds) {
        F.thr2 = 9.0f;
        return;
    }
    // cv2's LMeDSPointSetRegistrator: sigma = 2.5 * 1.4826 * (1 + 5 / (M - s)) * sqrt(median), at least 0.001
    const double med = (double)__uint_as_float((unsigned)(key >> 32));
    double sigma = __longlong_as_double(0x7ff0000000000000ll);
    if (F.M > s) sigma = DMUL(DMUL(DMUL(2.5, 1.4826), DADD(1.0, DDIV(5.0, (double)(F.M - s)))), __dsqrt_rn(med));
    sigma = fmax(sigma, 0.001);
    F.thr2 = __double2float_rn(DMUL(sigma, sigma));
}

// ------------------------------------------------------------------------------------------------ refinement
__device__ __forceinline__ bool is_inlier(const Frame& F, const Pt& q, bool lms, bool homog) {
    if (lms) return true;
    return (homog ? residual<true>(F.model, q) : residual<false>(F.model, q)) <= F.thr2;
}

template <int STAGE, int S>
__device__ __forceinline__ void accumulate(double (&acc)[S], const Frame& F, double X, double Y, double u, double v) {
    if (STAGE == kSim) {
        const double t[8] = {1.0, X, Y, X * X + Y * Y, X * u + Y * v, X * v - Y * u, u, v};
        for (int i = 0; i < 8; ++i) acc[i] += t[i];
    } else if (STAGE == kAff) {
        const double t[12] = {1.0, X, Y, X * X, X * Y, Y * Y, X * u, Y * u, u, X * v, Y * v, v};
        for (int i = 0; i < 12; ++i) acc[i] += t[i];
    } else if (STAGE == kCen) {
        const double t[5] = {1.0, X, Y, u, v};
        for (int i = 0; i < 5; ++i) acc[i] += t[i];
    } else if (STAGE == kMad) {
        acc[0] += fabs(X - F.cen[0]);
        acc[1] += fabs(Y - F.cen[1]);
        acc[2] += fabs(u - F.cen[2]);
        acc[3] += fabs(v - F.cen[3]);
    } else if (STAGE == kLtl) {
        const double Xn = (X - F.cen[0]) * F.scl[0], Yn = (Y - F.cen[1]) * F.scl[1];
        const double xn = (u - F.cen[2]) * F.scl[2], yn = (v - F.cen[3]) * F.scl[3];
        const double Lx[9] = {Xn, Yn, 1.0, 0.0, 0.0, 0.0, -xn * Xn, -xn * Yn, -xn};
        const double Ly[9] = {0.0, 0.0, 0.0, Xn, Yn, 1.0, -yn * Xn, -yn * Yn, -yn};
        int i = 0;
        for (int j = 0; j < 9; ++j)
            for (int k = j; k < 9; ++k) acc[i++] += Lx[j] * Lx[k] + Ly[j] * Ly[k];
    } else {
        const double* h = F.cand;
        const double iw = 1.0 / (h[6] * X + h[7] * Y + 1.0);
        const double px = (h[0] * X + h[1] * Y + h[2]) * iw, py = (h[3] * X + h[4] * Y + h[5]) * iw;
        const double ex = px - u, ey = py - v;
        const double Jx[8] = {X * iw, Y * iw, iw, 0.0, 0.0, 0.0, -px * X * iw, -px * Y * iw};
        const double Jy[8] = {0.0, 0.0, 0.0, X * iw, Y * iw, iw, -py * X * iw, -py * Y * iw};
        int i = 0;
        for (int j = 0; j < 8; ++j)
            for (int k = j; k < 8; ++k) acc[i++] += Jx[j] * Jx[k] + Jy[j] * Jy[k];
        for (int j = 0; j < 8; ++j) acc[36 + j] += Jx[j] * ex + Jy[j] * ey;
        acc[44] += ex * ex + ey * ey;
    }
}

// Per-block partial sums of a stage over the inliers of the frame, in coordinates centred on the frame centre.
template <int STAGE, bool HOMOG>
__global__ void __launch_bounds__(256) reduce_kernel(const float2* __restrict__ flow, const uint8_t* __restrict__ mask,
                                                     const Frame* __restrict__ fr, double* __restrict__ partials,
                                                     int H, int W, int ref, int bpf, int lms) {
    constexpr int S = stage_sums(STAGE);
    __shared__ double wsum[8][S];
    const size_t hw = (size_t)H * W, n = blockIdx.x / bpf, b = blockIdx.x - n * bpf;
    const Frame& F = fr[n];
    if (F.status != kFit) return;
    const double cx = 0.5 * (W - 1), cy = 0.5 * (H - 1);
    double acc[S];
#pragma unroll
    for (int i = 0; i < S; ++i) acc[i] = 0.0;
    for (int j = 0; j < kChunk / 256; ++j) {
        const size_t p = b * kChunk + j * 256 + threadIdx.x;
        if (p >= hw) break;
        if (mask && !mask[n * hw + p]) continue;
        const Pt q = make_point(flow + n * hw, p, W, ref);
        if (!is_inlier(F, q, lms, HOMOG)) continue;
        accumulate<STAGE, S>(acc, F, q.sx - cx, q.sy - cy, q.dx - cx, q.dy - cy);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < S; ++i) {
        double v = acc[i];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) wsum[wid][i] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < S; i += blockDim.x) {
        double t = wsum[0][i];
        for (int w = 1; w < 8; ++w) t += wsum[w][i];
        partials[(size_t)blockIdx.x * kMaxSums + i] = t;
    }
}

// Smallest eigenvector of a symmetric 9x9 matrix by cyclic Jacobi rotations.
__device__ void smallest_eigenvector(double (&a)[9][9], double (&vec)[9]) {
    double v[9][9];
    for (int i = 0; i < 9; ++i)
        for (int j = 0; j < 9; ++j) v[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 50; ++sweep) {
        double off = 0.0, all = 0.0;
        for (int p = 0; p < 9; ++p)
            for (int q = 0; q < 9; ++q) {
                all += a[p][q] * a[p][q];
                if (p != q) off += a[p][q] * a[p][q];
            }
        if (!(off > 1e-32 * all)) break;
        for (int p = 0; p < 8; ++p)
            for (int q = p + 1; q < 9; ++q) {
                if (a[p][q] == 0.0) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 9; ++k) {
                    const double akp = a[k][p], akq = a[k][q];
                    a[k][p] = c * akp - s * akq;
                    a[k][q] = s * akp + c * akq;
                }
                for (int k = 0; k < 9; ++k) {
                    const double apk = a[p][k], aqk = a[q][k];
                    a[p][k] = c * apk - s * aqk;
                    a[q][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < 9; ++k) {
                    const double vkp = v[k][p], vkq = v[k][q];
                    v[k][p] = c * vkp - s * vkq;
                    v[k][q] = s * vkp + c * vkq;
                }
            }
    }
    int m = 0;
    for (int i = 1; i < 9; ++i)
        if (a[i][i] < a[m][m]) m = i;
    for (int i = 0; i < 9; ++i) vec[i] = v[i][m];
}

// H (3x3, centred coordinates) -> pixel coordinates: T^-1 H T with T = translation by -(cx, cy); divided by H[2][2].
__device__ void uncentre(const double* hc, double cx, double cy, double* out) {
    double m1[9];
    for (int r = 0; r < 3; ++r) {
        m1[3 * r] = hc[3 * r];
        m1[3 * r + 1] = hc[3 * r + 1];
        m1[3 * r + 2] = hc[3 * r + 2] - cx * hc[3 * r] - cy * hc[3 * r + 1];
    }
    for (int c = 0; c < 3; ++c) {
        out[c] = m1[c] + cx * m1[6 + c];
        out[3 + c] = m1[3 + c] + cy * m1[6 + c];
        out[6 + c] = m1[6 + c];
    }
    const double d = out[8];
    for (int i = 0; i < 9; ++i) out[i] /= d;
}

// Solves the LM step from h with damping lambda: cand = h - (JtJ + lambda diag(JtJ))^-1 Jte; cand = h if singular.
__device__ void lm_candidate(Frame& F) {
    double A[8][8], b[8], x[8];
    int i = 0;
    for (int j = 0; j < 8; ++j)
        for (int k = j; k < 8; ++k, ++i) A[j][k] = A[k][j] = F.jtj[i];
    for (int j = 0; j < 8; ++j) {
        A[j][j] *= 1.0 + F.lambda;
        b[j] = -F.jte[j];
    }
    const bool ok = gauss_solve<8>(A, b, x);
    for (int j = 0; j < 8; ++j) F.cand[j] = ok ? F.h[j] + x[j] : F.h[j];
}

// One block per frame: the stage's sums over the frame's partials (fixed order), then the stage's arithmetic on thread
// 0. With last, every frame's results are written: identity (zero), NaN and count 0 (degenerate), or the fit.
template <int STAGE>
__global__ void __launch_bounds__(64) finish_kernel(Frame* __restrict__ fr, const double* __restrict__ partials,
                                                    int bpf, int H, int W, int iter, int last,
                                                    double* __restrict__ out_mats, int* __restrict__ out_counts) {
    constexpr int S = stage_sums(STAGE);
    __shared__ double sum[S];
    const size_t n = blockIdx.x;
    Frame& F = fr[n];
    if (F.status == kFit)
        for (int i = threadIdx.x; i < S; i += blockDim.x) {
            double t = 0.0;
            for (int b = 0; b < bpf; ++b) t += partials[(n * bpf + b) * kMaxSums + i];
            sum[i] = t;
        }
    __syncthreads();
    if (threadIdx.x != 0) return;
    const double cx = 0.5 * (W - 1), cy = 0.5 * (H - 1);
    double res[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (F.status == kFit) {
        if (STAGE == kSim || STAGE == kAff || STAGE == kCen) F.count = (int)sum[0];
        if (STAGE == kSim) {
            // rows (X, -Y, 1, 0) and (Y, X, 0, 1) for the parameters (a, b, tx, ty)
            const double n0 = sum[0], sX = sum[1], sY = sum[2], sR = sum[3];
            double A[4][4] = {{sR, 0.0, sX, sY}, {0.0, sR, -sY, sX}, {sX, -sY, n0, 0.0}, {sY, sX, 0.0, n0}};
            double b[4] = {sum[4], sum[5], sum[6], sum[7]}, x[4];
            if (F.count < 2 || !gauss_solve<4>(A, b, x)) {
                F.status = kDegenerate;
            } else {
                const double hc[9] = {x[0], -x[1], x[2], x[1], x[0], x[3], 0.0, 0.0, 1.0};
                uncentre(hc, cx, cy, res);
            }
        } else if (STAGE == kAff) {
            double hc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 1};
            bool ok = F.count >= 3;
            for (int r = 0; r < 2 && ok; ++r) {
                double A[3][3] = {{sum[3], sum[4], sum[1]}, {sum[4], sum[5], sum[2]}, {sum[1], sum[2], sum[0]}};
                double b[3] = {sum[6 + 3 * r], sum[7 + 3 * r], sum[8 + 3 * r]}, x[3];
                ok = gauss_solve<3>(A, b, x);
                hc[3 * r] = x[0], hc[3 * r + 1] = x[1], hc[3 * r + 2] = x[2];
            }
            if (ok) uncentre(hc, cx, cy, res);
            else F.status = kDegenerate;
        } else if (STAGE == kCen) {
            if (F.count < 4) F.status = kDegenerate;
            for (int i = 0; i < 4; ++i) F.cen[i] = sum[1 + i] / sum[0];
        } else if (STAGE == kMad) {
            for (int i = 0; i < 4; ++i) {
                if (fabs(sum[i]) < DBL_EPSILON) F.status = kDegenerate;
                F.scl[i] = F.count / sum[i];
            }
        } else if (STAGE == kLtl) {
            double a[9][9], v[9];
            int i = 0;
            for (int j = 0; j < 9; ++j)
                for (int k = j; k < 9; ++k, ++i) a[j][k] = a[k][j] = sum[i];
            smallest_eigenvector(a, v);
            // H = invHnorm(dst) * H0 * Hnorm(src) (cv2's HomographyEstimatorCallback::runKernel)
            const double sX = F.scl[0], sY = F.scl[1], tX = -F.cen[0] * F.scl[0], tY = -F.cen[1] * F.scl[1];
            double m[9];
            for (int r = 0; r < 3; ++r) {
                m[3 * r] = v[3 * r] * sX;
                m[3 * r + 1] = v[3 * r + 1] * sY;
                m[3 * r + 2] = v[3 * r] * tX + v[3 * r + 1] * tY + v[3 * r + 2];
            }
            const double ix = 1.0 / F.scl[2], iy = 1.0 / F.scl[3];
            double hc[9];
            for (int c = 0; c < 3; ++c) {
                hc[c] = ix * m[c] + F.cen[2] * m[6 + c];
                hc[3 + c] = iy * m[3 + c] + F.cen[3] * m[6 + c];
                hc[6 + c] = m[6 + c];
            }
            if (!(hc[8] != 0.0)) F.status = kDegenerate;
            for (int j = 0; j < 8; ++j) F.cand[j] = hc[j] / hc[8];
            if (!isfinite(F.cand[0])) F.status = kDegenerate;
        } else {
            const double e = sum[44];
            if (iter == 0 || e < F.err) {
                for (int j = 0; j < 8; ++j) F.h[j] = F.cand[j];
                for (int j = 0; j < 36; ++j) F.jtj[j] = sum[j];
                for (int j = 0; j < 8; ++j) F.jte[j] = sum[36 + j];
                F.err = e;
                F.lambda = fmax(F.lambda * 0.1, 1e-15);
                if (iter == 0 && !isfinite(e)) F.status = kDegenerate;
            } else {
                F.lambda *= 10.0;
            }
            if (!last) {
                lm_candidate(F);
            } else if (F.status == kFit) {
                const double hc[9] = {F.h[0], F.h[1], F.h[2], F.h[3], F.h[4], F.h[5], F.h[6], F.h[7], 1.0};
                uncentre(hc, cx, cy, res);
            }
        }
    }
    if (!last) return;
    if (F.status == kDegenerate) {
        for (int i = 0; i < 9; ++i) res[i] = __longlong_as_double(0x7ff8000000000000ll);
        F.count = 0;
    }
    if (F.status == kZero) F.count = 0;
    for (int i = 0; i < 9; ++i) out_mats[n * 9 + i] = res[i];
    if (out_counts) out_counts[n] = F.count;
}

template <bool HOMOG>
__global__ void __launch_bounds__(256) inliers_kernel(const float2* __restrict__ flow, const uint8_t* __restrict__ mask,
                                                      const Frame* __restrict__ fr, uint8_t* __restrict__ out,
                                                      size_t hw, int W, int ref, int lms, size_t total) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t n = i / hw, p = i - n * hw;
        const Frame& F = fr[n];
        uint8_t v = 0;
        if (F.status == kFit && (mask == nullptr || mask[i]))
            v = is_inlier(F, make_point(flow + n * hw, p, W, ref), lms, HOMOG);
        out[i] = v;
    }
}

// ------------------------------------------------------------------------------------------------ host side
static size_t pad256(size_t b) { return (b + 255) & ~size_t(255); }
static int chunks(size_t hw, int chunk) { return (int)((hw + chunk - 1) / chunk); }

struct Layout {
    size_t frames, flags, list, cnt, models, ok, counts, sel, hist, partials, total;
};

static Layout layout(int method, int K, int N, int H, int W) {
    const size_t hw = (size_t)H * W, bpf = chunks(hw, kChunk), nk = method == OFK_FIT_LMS ? 0 : (size_t)N * K;
    Layout L;
    size_t o = 0;
    L.frames = o, o += pad256(sizeof(Frame) * N);
    L.flags = o, o += pad256(sizeof(int) * N);
    L.list = o, o += pad256(sizeof(int) * N * hw);
    L.cnt = o, o += pad256(sizeof(int) * N * bpf);
    L.models = o, o += pad256(sizeof(double) * 9 * nk);
    L.ok = o, o += pad256(sizeof(int) * nk);
    L.counts = o, o += method == OFK_FIT_RANSAC ? pad256(sizeof(unsigned) * nk) : 0;
    L.sel = o, o += method == OFK_FIT_LMEDS ? pad256(sizeof(uint2) * nk) : 0;
    L.hist = o, o += method == OFK_FIT_LMEDS ? pad256(sizeof(unsigned) * kBins0 * nk) : 0;
    L.partials = o, o += pad256(sizeof(double) * kMaxSums * N * bpf);
    L.total = o;
    return L;
}

template <bool HOMOG>
static int run_scoring(const float2* flow, const uint8_t* mask, const Frame* fr, char* ws, const Layout& L, int method,
                       int K, int N, int H, int W, int ref, cudaStream_t st) {
    const int hw = H * W;
    const double* models = reinterpret_cast<const double*>(ws + L.models);
    const int* ok = reinterpret_cast<const int*>(ws + L.ok);
    const size_t nk = (size_t)N * K;
    if (method == OFK_FIT_RANSAC) {
        unsigned* counts = reinterpret_cast<unsigned*>(ws + L.counts);
        OFK_CUDA(cudaMemsetAsync(counts, 0, sizeof(unsigned) * nk, st));
        const int groups = (K + kCountG - 1) / kCountG, ch = chunks(hw, kCountChunk);
        score_kernel<HOMOG, -1><<<(unsigned)((size_t)N * groups * ch), 256, 0, st>>>(
            flow, mask, fr, models, ok, counts, nullptr, nullptr, K, hw, W, ref, groups, ch);
        OFK_LAUNCHED();
        return OFK_OK;
    }
    uint2* sel = reinterpret_cast<uint2*>(ws + L.sel);
    unsigned* hist = reinterpret_cast<unsigned*>(ws + L.hist);
    OFK_CUDA(cudaMemsetAsync(hist, 0, sizeof(unsigned) * kBins0 * nk, st));
    const int groups = (K + kHistG - 1) / kHistG, ch = chunks(hw, kHistChunk);
    const unsigned grid = (unsigned)((size_t)N * groups * ch), pgrid = (unsigned)((nk + 7) / 8);
    score_kernel<HOMOG, 0><<<grid, 256, 0, st>>>(flow, mask, fr, models, ok, nullptr, sel, hist, K, hw, W, ref, groups, ch);
    OFK_LAUNCHED();
    pick_kernel<0><<<pgrid, 256, 0, st>>>(fr, ok, sel, hist, K, nk);
    OFK_LAUNCHED();
    score_kernel<HOMOG, 1><<<grid, 256, 0, st>>>(flow, mask, fr, models, ok, nullptr, sel, hist, K, hw, W, ref, groups, ch);
    OFK_LAUNCHED();
    pick_kernel<1><<<pgrid, 256, 0, st>>>(fr, ok, sel, hist, K, nk);
    OFK_LAUNCHED();
    score_kernel<HOMOG, 2><<<grid, 256, 0, st>>>(flow, mask, fr, models, ok, nullptr, sel, hist, K, hw, W, ref, groups, ch);
    OFK_LAUNCHED();
    pick_kernel<2><<<pgrid, 256, 0, st>>>(fr, ok, sel, hist, K, nk);
    OFK_LAUNCHED();
    return OFK_OK;
}

template <int STAGE, bool HOMOG>
static int reduce_stage(const float2* flow, const uint8_t* mask, Frame* fr, double* partials, int N, int H, int W,
                        int ref, int lms, int iter, int last, double* out_mats, int* out_counts, cudaStream_t st) {
    const int bpf = chunks((size_t)H * W, kChunk);
    reduce_kernel<STAGE, HOMOG><<<(unsigned)((size_t)N * bpf), 256, 0, st>>>(flow, mask, fr, partials, H, W, ref, bpf,
                                                                            lms);
    OFK_LAUNCHED();
    finish_kernel<STAGE><<<N, 64, 0, st>>>(fr, partials, bpf, H, W, iter, last, out_mats, out_counts);
    OFK_LAUNCHED();
    return OFK_OK;
}

#define OFK_TRY(call)                 \
    do {                              \
        const int rc_ = (call);       \
        if (rc_ != OFK_OK) return rc_; \
    } while (0)

template <bool HOMOG>
static int refine(const float2* flow, const uint8_t* mask, Frame* fr, double* partials, int dof, int lms, int N, int H,
                  int W, int ref, double* out_mats, int* out_counts, cudaStream_t st) {
    if constexpr (!HOMOG) {
        if (dof == 4) return reduce_stage<kSim, false>(flow, mask, fr, partials, N, H, W, ref, lms, 0, 1, out_mats, out_counts, st);
        return reduce_stage<kAff, false>(flow, mask, fr, partials, N, H, W, ref, lms, 0, 1, out_mats, out_counts, st);
    } else {
        OFK_TRY((reduce_stage<kCen, true>(flow, mask, fr, partials, N, H, W, ref, lms, 0, 0, nullptr, nullptr, st)));
        OFK_TRY((reduce_stage<kMad, true>(flow, mask, fr, partials, N, H, W, ref, lms, 0, 0, nullptr, nullptr, st)));
        OFK_TRY((reduce_stage<kLtl, true>(flow, mask, fr, partials, N, H, W, ref, lms, 0, 0, nullptr, nullptr, st)));
        for (int it = 0; it <= kLmIters; ++it)
            OFK_TRY((reduce_stage<kLm, true>(flow, mask, fr, partials, N, H, W, ref, lms, it, it == kLmIters, out_mats,
                                             out_counts, st)));
        return OFK_OK;
    }
}

template <bool HOMOG>
static int run_fit(const float* flow_f, const uint8_t* mask, int ref, int dof, int method, int K, float thr,
                   double* out_mats, uint8_t* out_inliers, int* out_counts, int N, int H, int W, char* ws,
                   const Layout& L, cudaStream_t st) {
    const float2* flow = reinterpret_cast<const float2*>(flow_f);
    const size_t hw = (size_t)H * W;
    const int s = dof / 2, bpf = chunks(hw, kChunk), lms = method == OFK_FIT_LMS;
    Frame* fr = reinterpret_cast<Frame*>(ws + L.frames);
    int* flags = reinterpret_cast<int*>(ws + L.flags);
    int* list = mask ? reinterpret_cast<int*>(ws + L.list) : nullptr;
    int* cnt = reinterpret_cast<int*>(ws + L.cnt);
    double* models = reinterpret_cast<double*>(ws + L.models);
    int* ok = reinterpret_cast<int*>(ws + L.ok);
    OFK_TRY(ofk_nonzero_flags(flow_f, mask, thr, flags, N, H, W, reinterpret_cast<ofk_stream_t>(st)));
    if (list) {
        list_count_kernel<<<(unsigned)((size_t)N * bpf), 256, 0, st>>>(mask, cnt, hw, bpf);
        OFK_LAUNCHED();
    }
    frames_kernel<<<(N + 127) / 128, 128, 0, st>>>(flags, cnt, fr, N, (int)hw, bpf, list != nullptr, s);
    OFK_LAUNCHED();
    if (list) {
        list_scatter_kernel<<<(unsigned)((size_t)N * bpf), 256, 0, st>>>(mask, cnt, list, hw, bpf);
        OFK_LAUNCHED();
    }
    if (!lms) {
        const size_t nk = (size_t)N * K;
        const unsigned grid = (unsigned)((nk + 127) / 128);
        if (dof == 4) hypotheses_kernel<4><<<grid, 128, 0, st>>>(flow, list, fr, models, ok, K, nk, (int)hw, W, ref);
        else if (dof == 6) hypotheses_kernel<6><<<grid, 128, 0, st>>>(flow, list, fr, models, ok, K, nk, (int)hw, W, ref);
        else hypotheses_kernel<8><<<grid, 128, 0, st>>>(flow, list, fr, models, ok, K, nk, (int)hw, W, ref);
        OFK_LAUNCHED();
        OFK_TRY(run_scoring<HOMOG>(flow, mask, fr, ws, L, method, K, N, H, W, ref, st));
        select_kernel<<<N, 256, 0, st>>>(fr, models, ok, reinterpret_cast<const unsigned*>(ws + L.counts),
                                         reinterpret_cast<const uint2*>(ws + L.sel), K, method == OFK_FIT_LMEDS, s);
        OFK_LAUNCHED();
    }
    OFK_TRY(refine<HOMOG>(flow, mask, fr, reinterpret_cast<double*>(ws + L.partials), dof, lms, N, H, W, ref, out_mats,
                          out_counts, st));
    if (out_inliers) {
        const size_t total = (size_t)N * hw;
        const size_t blocks = std::min((total + 255) / 256, (size_t)sm_count() * 32);
        inliers_kernel<HOMOG><<<(unsigned)blocks, 256, 0, st>>>(flow, mask, fr, out_inliers, hw, W, ref, lms, total);
        OFK_LAUNCHED();
    }
    return OFK_OK;
}

// Blocks of the largest grid (scoring) per frame; N times this must stay within grid x.
static size_t score_blocks_per_frame(int method, int K, size_t hw) {
    if (method == OFK_FIT_RANSAC) return (size_t)((K + kCountG - 1) / kCountG) * chunks(hw, kCountChunk);
    if (method == OFK_FIT_LMEDS) return (size_t)((K + kHistG - 1) / kHistG) * chunks(hw, kHistChunk);
    return chunks(hw, kChunk);
}

}  // namespace fit
}  // namespace ofk

using namespace ofk;

static bool fit_args_ok(int dof, int method, int hypotheses, int N, int H, int W) {
    return (dof == 4 || dof == 6 || dof == 8) && (method == OFK_FIT_RANSAC || method == OFK_FIT_LMEDS ||
                                                  (method == OFK_FIT_LMS && dof == 8)) &&
           hypotheses >= 1 && hypotheses <= 65536 && N >= 0 && N <= 65535 && H > 0 && W > 0 &&
           (size_t)H * W < (1ull << 31);
}

extern "C" size_t ofk_fit_matrix_workspace(int dof, int method, int hypotheses, int N, int H, int W) {
    if (!fit_args_ok(dof, method, hypotheses, N, H, W)) return 0;
    return fit::layout(method, hypotheses, N, H, W).total;
}

extern "C" int ofk_fit_matrix(const float* flow, const uint8_t* mask, int ref, int dof, int method, int hypotheses,
                              float thr, int masked, double* out_mats, uint8_t* out_inliers, int* out_counts, int N,
                              int H, int W, void* ws, size_t ws_bytes, ofk_stream_t stream) {
    OFK_CHECK_ARG(flow && out_mats && ws, "ofk_fit_matrix: NULL pointer");
    OFK_CHECK_ARG(ref == 's' || ref == 't', "ofk_fit_matrix: ref must be 's' or 't'");
    OFK_CHECK_ARG(dof == 4 || dof == 6 || dof == 8, "ofk_fit_matrix: dof must be 4, 6 or 8, got %d", dof);
    OFK_CHECK_ARG(method == OFK_FIT_RANSAC || method == OFK_FIT_LMEDS || method == OFK_FIT_LMS,
                  "ofk_fit_matrix: method must be OFK_FIT_LMS, OFK_FIT_RANSAC or OFK_FIT_LMEDS");
    OFK_CHECK_ARG(method != OFK_FIT_LMS || dof == 8, "ofk_fit_matrix: OFK_FIT_LMS needs dof 8");
    OFK_CHECK_ARG(hypotheses >= 1 && hypotheses <= 65536, "ofk_fit_matrix: hypotheses must be in [1, 65536], got %d",
                  hypotheses);
    OFK_CHECK_ARG(N >= 0 && N <= 65535 && H > 0 && W > 0 && (size_t)H * W < (1ull << 31),
                  "ofk_fit_matrix: bad shape N=%d H=%d W=%d (N <= 65535, H*W < 2^31)", N, H, W);
    OFK_CHECK_ARG(thr >= 0.f, "ofk_fit_matrix: thr must be >= 0");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(flow) & 7) == 0, "ofk_fit_matrix: flow must be 8-byte aligned");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(ws) & 7) == 0, "ofk_fit_matrix: ws must be 8-byte aligned");
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(out_mats) & 7) == 0 && (reinterpret_cast<uintptr_t>(out_counts) & 3) == 0,
                  "ofk_fit_matrix: out_mats must be 8-byte and out_counts 4-byte aligned");
    const size_t need = fit::layout(method, hypotheses, N, H, W).total;
    OFK_CHECK_ARG(ws_bytes >= need, "ofk_fit_matrix: workspace too small (%zu bytes, need %zu)", ws_bytes, need);
    OFK_CHECK_ARG((size_t)N * fit::score_blocks_per_frame(method, hypotheses, (size_t)H * W) <= 0x7fffffffu,
                  "ofk_fit_matrix: batch too large for one call (N=%d, %d hypotheses, H=%d W=%d)", N, hypotheses, H, W);
    if (N == 0) return OFK_OK;
    const fit::Layout L = fit::layout(method, hypotheses, N, H, W);
    const uint8_t* m = masked ? mask : nullptr;
    char* w = static_cast<char*>(ws);
    cudaStream_t st = as_stream(stream);
    if (dof == 8)
        return fit::run_fit<true>(flow, m, ref, dof, method, hypotheses, thr, out_mats, out_inliers, out_counts, N, H, W,
                                  w, L, st);
    return fit::run_fit<false>(flow, m, ref, dof, method, hypotheses, thr, out_mats, out_inliers, out_counts, N, H, W,
                               w, L, st);
}
