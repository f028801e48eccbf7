// Source-referenced (forward) resampling for sm_100a: replaces scipy.interpolate.griddata(points = grid + flow,
// values, grid, 'linear') + nan_to_num at utils.py:237-258 of the reference (Flow.apply ref 's', same-reference
// invert, switch_ref, combine modes 1 / 2, the 's'-side valid areas).
//
// griddata triangulates the displaced pixel positions (Qhull Delaunay, AFTER dropping the points a `consider_mask`
// removes) and interpolates barycentrically inside each triangle, 0 outside the convex hull. The algorithm and its
// predicates live in forward_geom.cuh / forward_irregular.cuh (shared with the host build the CPU tests run against
// the reference's goldens); this file maps it onto the GPU:
//
//   fwd_raster_kernel   regular part. A CTA owns a tile of 64 x 16 source cells: the 65 x 17 displaced vertices
//                       (float64 positions, computed once per vertex), their payload and mask bytes are staged in
//                       shared memory; one thread per cell column walks 4 rows keeping the shared row of vertices in
//                       registers, picks the Delaunay diagonal and rasterises both triangles. The fill rule makes every
//                       pixel inside the mesh the product of exactly one triangle, so values and validity go straight
//                       to the output: no triangle-id plane in HBM, no atomics, no second pass over the frame.
//   irr_*               irregular part: pixels no intact cell produced (marker byte left in the validity plane) are
//                       located in the Delaunay triangulation of the boundary sites (frame border, rims of removed
//                       points), binned by position with two counting passes and a scan; a per-frame hull polygon
//                       rejects the pixels outside the hull without a search.
//   legacy::fwd_scatter / fwd_gather   folding fields (a displaced cell with a non-positive triangle): several
//                       triangles cover a pixel, "exactly one" no longer holds; such frames are redone completely by
//                       the order-independent atomicMax(triangle id) resolve of round 1 (largest source index wins).
//
// Deviation left (DESIGN.md): cells whose four corners are co-circular to within rounding have no unique Delaunay
// diagonal (similarity transforms of the pixel grid); Qhull's pick there is an artefact of its facet merging.
#include <algorithm>

#include <mutex>

#include "ofk_common.cuh"
#include "forward_irregular.cuh"
#include "track_device.cuh"

// ============================================================ order-independent resolve for folding fields (round 1)
namespace ofk {
namespace legacy {

struct P2 {
    double x, y;
};

__device__ __forceinline__ P2 displaced(const float2* __restrict__ fl, int W, int row, int col, float sign) {
    const float2 f = __ldg(fl + row * W + col);
    P2 p;
    p.x = static_cast<double>(col) + static_cast<double>(sign * f.x);
    p.y = static_cast<double>(row) + static_cast<double>(sign * f.y);
    return p;
}

__device__ __forceinline__ double orient(const P2& a, const P2& b, const P2& c) {
    return (b.x - a.x) * (c.y - a.y) - (b.y - a.y) * (c.x - a.x);
}

// > 0 iff d lies inside the circumcircle of the positively oriented triangle (a, b, c)
__device__ __forceinline__ double incircle(const P2& a, const P2& b, const P2& c, const P2& d) {
    const double ax = a.x - d.x, ay = a.y - d.y, bx = b.x - d.x, by = b.y - d.y, cx = c.x - d.x, cy = c.y - d.y;
    const double a2 = ax * ax + ay * ay, b2 = bx * bx + by * by, c2 = cx * cx + cy * cy;
    return ax * (by * c2 - b2 * cy) - ay * (bx * c2 - b2 * cx) + a2 * (bx * cy - by * cx);
}

// Corner naming of cell (i, j): a = (i, j), b = (i, j+1), c = (i+1, j), d = (i+1, j+1).
// diag 0 splits along a-d: triangles (a, b, d) and (a, d, c); diag 1 along b-c: (a, b, c) and (b, d, c).
__device__ __forceinline__ int choose_diagonal(const P2& a, const P2& b, const P2& c, const P2& d,
                                               double flip_tol = 0.0) {
    const double o0a = orient(a, b, d), o0b = orient(a, d, c);   // diag 0 halves
    const double o1a = orient(a, b, c), o1b = orient(b, d, c);   // diag 1 halves
    const bool ok0 = (o0a > 0 && o0b > 0) || (o0a < 0 && o0b < 0);
    const bool ok1 = (o1a > 0 && o1b > 0) || (o1a < 0 && o1b < 0);
    if (ok0 && ok1) {  // convex quad: Delaunay criterion
        const double det = incircle(a, b, d, c);
        const bool c_inside = (o0a > 0) ? (det > 0) : (det < 0);
        return (c_inside ? 1 : 0) ^ (fabs(det) <= flip_tol ? 1 : 0);   // flip_tol: test hook, see cell_diagonal
    }
    return ok1 && !ok0 ? 1 : 0;
}

// vertex k (0..2) of triangle `tri` (0/1) of a cell split by `diag`, as corner code 0=a 1=b 2=c 3=d
__device__ __forceinline__ int corner_of(int diag, int tri, int k) {
    // diag0: t0 = a b d, t1 = a d c ; diag1: t0 = a b c, t1 = b d c
    const int table = diag == 0 ? (tri == 0 ? 0x310 : 0x230) : (tri == 0 ? 0x210 : 0x231);
    return (table >> (4 * k)) & 0xf;
}

// Edge function of pixel q against edge (u, v), evaluated with the endpoints in canonical (index) order so the two
// triangles sharing an edge see bit-identical magnitudes with opposite signs.
__device__ __forceinline__ double edge_fn(const P2& u, int iu, const P2& v, int iv, double qx, double qy) {
    if (iu < iv) return (v.x - u.x) * (qy - u.y) - (v.y - u.y) * (qx - u.x);
    return -((u.x - v.x) * (qy - v.y) - (u.y - v.y) * (qx - v.x));
}

__device__ __forceinline__ void scatter_tile(const float* __restrict__ flow, float sign,
                                             const uint8_t* __restrict__ point_mask,
                                             unsigned int* __restrict__ winner, int H, int W, int bx, int by, int n) {
    const int j = bx * 32 + (threadIdx.x & 31);
    const int i = by * 8 + (threadIdx.x >> 5);
    if (i >= H - 1 || j >= W - 1) return;
    const size_t fbase = (size_t)n * H * W;
    const float2* fl = reinterpret_cast<const float2*>(flow) + fbase;
    if (point_mask != nullptr) {
        const uint8_t* pm = point_mask + fbase;
        const int o = i * W + j;
        if (!(pm[o] && pm[o + 1] && pm[o + W] && pm[o + W + 1])) return;
    }
    P2 v[4];
    v[0] = displaced(fl, W, i, j, sign);
    v[1] = displaced(fl, W, i, j + 1, sign);
    v[2] = displaced(fl, W, i + 1, j, sign);
    v[3] = displaced(fl, W, i + 1, j + 1, sign);
    const int vid[4] = {i * W + j, i * W + j + 1, (i + 1) * W + j, (i + 1) * W + j + 1};
    const int diag = choose_diagonal(v[0], v[1], v[2], v[3]);
    unsigned int* win = winner + fbase;
#pragma unroll
    for (int tri = 0; tri < 2; ++tri) {
        const int c0 = corner_of(diag, tri, 0), c1 = corner_of(diag, tri, 1), c2 = corner_of(diag, tri, 2);
        const P2 p0 = v[c0], p1 = v[c1], p2 = v[c2];
        const double area2 = orient(p0, p1, p2);
        if (area2 == 0.0) continue;
        const double sgn = area2 > 0 ? 1.0 : -1.0;
        // candidate pixels: bounding box in float32, rounded outwards (a superset is enough: coverage is decided by
        // the exact edge functions below)
        int xmin = (int)ceilf(fminf(__double2float_rd(p0.x), fminf(__double2float_rd(p1.x), __double2float_rd(p2.x))));
        int xmax = (int)floorf(fmaxf(__double2float_ru(p0.x), fmaxf(__double2float_ru(p1.x), __double2float_ru(p2.x))));
        int ymin = (int)ceilf(fminf(__double2float_rd(p0.y), fminf(__double2float_rd(p1.y), __double2float_rd(p2.y))));
        int ymax = (int)floorf(fmaxf(__double2float_ru(p0.y), fmaxf(__double2float_ru(p1.y), __double2float_ru(p2.y))));
        xmin = max(xmin, 0);
        ymin = max(ymin, 0);
        xmax = min(xmax, W - 1);
        ymax = min(ymax, H - 1);
        const unsigned int id = ((unsigned int)(i * W + j) << 2 | (unsigned int)(tri << 1) | (unsigned int)diag) + 1u;
        for (int y = ymin; y <= ymax; ++y) {
            for (int x = xmin; x <= xmax; ++x) {
                const double qx = x, qy = y;
                const double e0 = sgn * edge_fn(p1, vid[c1], p2, vid[c2], qx, qy);
                const double e1 = sgn * edge_fn(p2, vid[c2], p0, vid[c0], qx, qy);
                const double e2 = sgn * edge_fn(p0, vid[c0], p1, vid[c1], qx, qy);
                if (e0 >= 0.0 && e1 >= 0.0 && e2 >= 0.0) atomicMax(win + y * W + x, id);
            }
        }
    }
}

// The resolve kernels run on small grids that loop over the tiles of the frames flagged as folded: for every other
// frame (the normal case) a launch costs a few hundred empty CTAs instead of one per tile.
__global__ void __launch_bounds__(256, 4) fwd_scatter(const float* __restrict__ flow, float sign,
                                                   const uint8_t* __restrict__ point_mask,
                                                   unsigned int* __restrict__ winner, int H, int W,
                                                   const int* __restrict__ folded) {
    const int n = blockIdx.y;
    if (folded[n] != 1) return;
    const int tx = (W - 1 + 31) / 32, ty = (H - 1 + 7) / 8;
    for (int t = blockIdx.x; t < tx * ty; t += gridDim.x) scatter_tile(flow, sign, point_mask, winner, H, W, t % tx, t / tx, n);
}

__device__ __forceinline__ void gather_tile(const float* __restrict__ payload, int C,
                                            const float* __restrict__ flow, float sign,
                                            const uint8_t* __restrict__ payload_mask,
                                            const unsigned int* __restrict__ winner, float* __restrict__ out,
                                            uint8_t* __restrict__ out_mask, int rule, int H, int W,
                                            unsigned long long inv_w /* ceil(2^64 / W) */, int bx, int by, int n) {
    const int x = bx * 32 + (threadIdx.x & 31);
    const int y = by * 8 + (threadIdx.x >> 5);
    if (x >= W || y >= H) return;
    const size_t fbase = (size_t)n * H * W;
    const int pix = y * W + x;
    const unsigned int id = winner[fbase + pix];
    if (id == 0u) {
        for (int c = 0; c < C; ++c) out[(fbase + pix) * C + c] = 0.f;
        if (out_mask) out_mask[fbase + pix] = 0;
        return;
    }
    const unsigned int code = id - 1u;
    const int diag = code & 1, tri = (code >> 1) & 1, cell = (int)(code >> 2);
    const int i = (int)__umul64hi((unsigned long long)cell, inv_w), j = cell - i * W;   // exact: cell < 2^29
    const float2* fl = reinterpret_cast<const float2*>(flow) + fbase;
    int vidx[3];
    P2 p[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int c = corner_of(diag, tri, k);
        const int r = i + (c >> 1), q = j + (c & 1);
        vidx[k] = r * W + q;
        p[k] = displaced(fl, W, r, q, sign);
    }
    const double area2 = orient(p[0], p[1], p[2]);
    const double qx = x, qy = y;
    // one reciprocal instead of two divisions: the weights move by an ulp at most (values are compared at 1e-3, the
    // mask tests below are decided by exact zeros and by margins far above an ulp)
    const double inv_area = __drcp_rn(area2);
    double w0 = edge_fn(p[1], vidx[1], p[2], vidx[2], qx, qy) * inv_area;
    double w1 = edge_fn(p[2], vidx[2], p[0], vidx[0], qx, qy) * inv_area;
    double w2 = 1.0 - w0 - w1;
    const float* pay = payload + fbase * C;
    for (int c = 0; c < C; ++c) {
        const double val = w0 * (double)__ldg(pay + (size_t)vidx[0] * C + c) +
                           w1 * (double)__ldg(pay + (size_t)vidx[1] * C + c) +
                           w2 * (double)__ldg(pay + (size_t)vidx[2] * C + c);
        out[(fbase + pix) * C + c] = (float)val;
    }
    if (out_mask) {
        double m = w0 + w1 + w2;
        if (payload_mask) {
            const uint8_t* pm = payload_mask + fbase;
            m = (pm[vidx[0]] ? w0 : 0.0) + (pm[vidx[1]] ? w1 : 0.0) + (pm[vidx[2]] ? w2 : 0.0);
        }
        bool ok;
        if (rule == OFK_RULE_STRICT) ok = ((float)m == 1.0f);   // float payloads: `== 1` after the float32 cast
        else ok = (m > 0.5);                                    // integer payloads: np.round(m) == 1
        out_mask[fbase + pix] = ok ? 1 : 0;
    }
}


__global__ void __launch_bounds__(256) fwd_gather(const float* __restrict__ payload, int C,
                                                  const float* __restrict__ flow, float sign,
                                                  const uint8_t* __restrict__ payload_mask,
                                                  const unsigned int* __restrict__ winner, float* __restrict__ out,
                                                  uint8_t* __restrict__ out_mask, int rule, int H, int W,
                                                  unsigned long long inv_w, const int* __restrict__ folded) {
    const int n = blockIdx.y;
    if (folded[n] != 1) return;
    const int tx = (W + 31) / 32, ty = (H + 7) / 8;
    for (int t = blockIdx.x; t < tx * ty; t += gridDim.x)
        gather_tile(payload, C, flow, sign, payload_mask, winner, out, out_mask, rule, H, W, inv_w, t % tx, t / tx, n);
}

__global__ void __launch_bounds__(256) fwd_clear(unsigned int* __restrict__ winner, size_t frame_px,
                                                 const int* __restrict__ folded) {
    const int n = blockIdx.y;
    if (folded[n] != 1) return;
    for (size_t t = (size_t)blockIdx.x * 256 + threadIdx.x; t < frame_px; t += (size_t)gridDim.x * 256)
        winner[(size_t)n * frame_px + t] = 0u;
}

}  // namespace legacy
}  // namespace ofk

// =========================================================================================== the B200 pipeline
namespace ofk {
namespace fwdk {
using namespace fwd;

__device__ unsigned long long g_stats[8];   // located, outside (by search), failed walks, rejected by the hull filter,
                                            // pixels handed to the pocket pass, its work items

constexpr int TW = 64, TH = 16, SW = TW + 1, SH = TH + 1, NV = SW * SH;
constexpr uint8_t UNCOVERED = 0xFF;

struct RasterArgs {
    const float* payload;
    const float* flow;
    const uint8_t* payload_mask;
    const uint8_t* point_mask;
    float* out;
    uint8_t* out_mask;
    uint8_t* cover;      // == out_mask when the caller wants the validity plane, else a workspace plane
    int* folded;
    float sign;
    int C, rule_strict, H, W;
    double flip_tol;     // test hook, 0 in production (see cell_diagonal)
};

template <int CT>
struct EmitDev {
    const RasterArgs& A;
    const float* s_pay;
    const uint8_t* s_pm;
    int sbase;           // shared-memory index of corner a
    size_t frame;        // n * H * W
    int gi, gj;          // cell
    __device__ __forceinline__ void operator()(int x, int y, int k0, int k1, int k2, double w0, double w1,
                                               double w2) const {
        const int v0 = sbase + (k0 >> 1) * SW + (k0 & 1), v1 = sbase + (k1 >> 1) * SW + (k1 & 1),
                  v2 = sbase + (k2 >> 1) * SW + (k2 & 1);
        const size_t px = frame + (size_t)y * A.W + x;
        const bool m0 = s_pm[v0] != 0, m1 = s_pm[v1] != 0, m2 = s_pm[v2] != 0;
        if (CT >= 0) {
            constexpr int C = CT > 0 ? CT : 0;
            interp_store(s_pay + v0 * C, s_pay + v1 * C, s_pay + v2 * C, m0, m1, m2, w0, w1, w2, C, A.out + px * C,
                         A.out_mask ? A.out_mask + px : nullptr, A.rule_strict);
        } else {
            const size_t g0 = frame + (size_t)(gi + (k0 >> 1)) * A.W + gj + (k0 & 1),
                         g1 = frame + (size_t)(gi + (k1 >> 1)) * A.W + gj + (k1 & 1),
                         g2 = frame + (size_t)(gi + (k2 >> 1)) * A.W + gj + (k2 & 1);
            interp_store(A.payload + g0 * A.C, A.payload + g1 * A.C, A.payload + g2 * A.C, m0, m1, m2, w0, w1, w2, A.C,
                         A.out + px * A.C, A.out_mask ? A.out_mask + px : nullptr, A.rule_strict);
        }
        if (A.out_mask == nullptr) A.cover[px] = 1;
    }
};

// ---- float32 helpers of the raster kernel (filters only: every decision they cannot take with a safety margin is
// ---- taken by the float64 predicates of forward_geom.cuh, so the result is the one of the host build)
__device__ __forceinline__ float edgef(const float2& u, const float2& v, float qx, float qy) {
    return (v.x - u.x) * (qy - u.y) - (v.y - u.y) * (qx - u.x);
}
__device__ __forceinline__ float orientf(const float2& a, const float2& b, const float2& c) {
    return (b.x - a.x) * (c.y - a.y) - (b.y - a.y) * (c.x - a.x);
}
// round-to-nearest integer of |v| < 2^22 without the conversion pipe
__device__ __forceinline__ int rint_magic(float v) { return __float_as_int(v + 12582912.0f) - 0x4B400000; }
__device__ __forceinline__ float int_to_float_magic(int i) { return __int_as_float(i + 0x4B400000) - 12582912.0f; }
__device__ __forceinline__ int floor_magic(float v) {
    const int r = rint_magic(v);
    return r - (int_to_float_magic(r) > v ? 1 : 0);
}
__device__ __forceinline__ int ceil_magic(float v) {
    const int r = rint_magic(v);
    return r + (int_to_float_magic(r) < v ? 1 : 0);
}

constexpr int QCAP = 256;          // candidate ring per warp (records), power of two
constexpr int REC_OK = 1 << 15;    // record flag: the cell is a positively oriented convex quadrilateral (float32 proof)

// Tile kernel. Phase 1 (one thread per cell column, rows of the warp's strip in turn): float32 bounding box of the
// displaced cell -> the candidate pixels (1.3 per cell for rotation-like fields) go into the warp's ring; a folded cell
// sets the frame's flag. Phase 2 (whenever 32 candidates are queued): one candidate per lane -- float32 edge functions
// reject or accept it (exact float64 evaluation only inside a rounding margin), the Delaunay diagonal by the float64
// in-circle determinant, weights and payload in float64. Without the queue the 1..4 candidates of a cell are a
// divergent loop that runs its longest trip count on every warp (measured: 765 thread instructions per pixel).
template <int CT>
#ifndef OFK_RASTER_CTAS
#define OFK_RASTER_CTAS 3
#endif
__global__ void __launch_bounds__(256, OFK_RASTER_CTAS) fwd_raster_kernel(const RasterArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int PC = CT > 0 ? CT : 0;
    P2* s_pos = reinterpret_cast<P2*>(smem);
    float2* s_posf = reinterpret_cast<float2*>(s_pos + NV);
    float* s_pay = reinterpret_cast<float*>(s_posf + NV);
    uint2* s_q = reinterpret_cast<uint2*>(s_pay + NV * PC + ((NV * PC) & 1));
    uint8_t* s_pm = reinterpret_cast<uint8_t*>(s_q + 8 * QCAP);
    uint8_t* s_pt = s_pm + NV;
    const int n = blockIdx.z, i0 = blockIdx.y * TH, j0 = blockIdx.x * TW;
    const size_t frame = (size_t)n * A.H * A.W;
    const float2* fl = reinterpret_cast<const float2*>(A.flow) + frame;
    // Staging: every global load of the tile (frame state, centre vertex, the thread's <= 5 vertices with payload and
    // mask bytes) is requested before the first one is used -- one memory round trip per CTA instead of one per loop
    // trip plus two dependent ones in front (ncu: half of the kernel's stall samples sat on these loads).
    constexpr int VPT = (NV + 255) / 256;
    const int fstate = A.folded[n];   // 2 = passed through (set by an earlier kernel); other CTAs may store 1 meanwhile
    const int cgi = min(i0 + TH / 2, A.H - 1), cgj = min(j0 + TW / 2, A.W - 1);
    const float2 fc = __ldg(fl + (size_t)cgi * A.W + cgj);
    float2 fv[VPT];
    float pay[VPT][PC > 0 ? PC : 1];
    uint8_t pmv[VPT], ptv[VPT];
#pragma unroll
    for (int k = 0; k < VPT; ++k) {
        const int v = min((int)threadIdx.x + k * 256, NV - 1);   // (the clamped duplicates are not stored)
        const int r = v / SW, c = v - r * SW;
        const int gi = min(i0 + r, A.H - 1), gj = min(j0 + c, A.W - 1);
        const size_t g = (size_t)gi * A.W + gj;
        fv[k] = __ldg(fl + g);
#pragma unroll
        for (int q = 0; q < PC; ++q) pay[k][q] = __ldg(A.payload + (frame + g) * PC + q);
        pmv[k] = A.payload_mask ? __ldg(A.payload_mask + frame + g) : (uint8_t)1;
        ptv[k] = A.point_mask ? __ldg(A.point_mask + frame + g) : (uint8_t)1;
    }
    if (fstate == 2) return;   // passed through (zero flow)
    // pixel origin of the tile's local float32 coordinates: the displaced centre vertex
    int ox, oy;
    {
        const P2 pc = displaced(fc.x, fc.y, cgi, cgj, A.sign);
        ox = (int)fmin(fmax(rint(pc.x), -1048576.0), 1048576.0);
        oy = (int)fmin(fmax(rint(pc.y), -1048576.0), 1048576.0);
    }
#pragma unroll
    for (int k = 0; k < VPT; ++k) {
        const int v = (int)threadIdx.x + k * 256;
        if (v < NV) {
            const int r = v / SW, c = v - r * SW;
            const int gi = min(i0 + r, A.H - 1), gj = min(j0 + c, A.W - 1);
            const P2 p = displaced(fv[k].x, fv[k].y, gi, gj, A.sign);
            s_pos[v] = p;
            s_posf[v] = make_float2((float)(p.x - (double)ox), (float)(p.y - (double)oy));
#pragma unroll
            for (int q = 0; q < PC; ++q) s_pay[v * PC + q] = pay[k][q];
            s_pm[v] = pmv[k];
            s_pt[v] = ptv[k];
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // warp w: columns (w & 1) * 32 .. + 31, rows (w >> 1) * 4 .. + 3 of the tile
    const int jl = (warp & 1) * 32 + lane, ilbase = (warp >> 1) * (TH / 4);
    const int gj = j0 + jl;
    uint2* q = s_q + warp * QCAP;
    unsigned head = 0, tail = 0;
    const float lxmin = (float)(0 - ox), lxmax = (float)(A.W - 1 - ox), lymin = (float)(0 - oy),
                lymax = (float)(A.H - 1 - oy);

    // ---------------------------------------------------------------- phase 2: one queued candidate per lane
    auto drain = [&](unsigned count) {
        const bool have = lane < count;
        const uint2 rec = have ? q[(head + lane) & (QCAP - 1)] : make_uint2(0u, 0u);
        head += count;
        if (!have) return;
        const int sb = rec.x & 0x7fff;
        const bool convex_ok = (rec.x & REC_OK) != 0;
        const int x = rec.y & 0xffff, y = rec.y >> 16;
        const float qxf = int_to_float_magic(x - ox), qyf = int_to_float_magic(y - oy);
        const float2 af = s_posf[sb], bf = s_posf[sb + 1], cf = s_posf[sb + SW], df = s_posf[sb + SW + 1];
        const float fab = edgef(af, bf, qxf, qyf), fbd = edgef(bf, df, qxf, qyf), fcd = edgef(cf, df, qxf, qyf),
                    fac = edgef(af, cf, qxf, qyf);
        // rounding margin of a float32 edge function: positions carry half an ulp of their magnitude
        const float mag = fmaxf(fmaxf(fabsf(af.x), fabsf(af.y)), fmaxf(fabsf(df.x), fabsf(df.y))) + 4.0f;
        const float ext = fabsf(df.x - af.x) + fabsf(df.y - af.y) + fabsf(bf.x - cf.x) + fabsf(bf.y - cf.y) + 2.0f;
        const float m = 1e-6f * mag * ext;
        bool decided = convex_ok && fabsf(fab) > m && fabsf(fbd) > m && fabsf(fcd) > m && fabsf(fac) > m;
        if (decided && !(fab > 0 && fbd > 0 && fcd < 0 && fac < 0)) return;   // outside the cell
        const P2 a = s_pos[sb], b = s_pos[sb + 1], c = s_pos[sb + SW], d = s_pos[sb + SW + 1];
        const double qx = (double)x, qy = (double)y;
        int diag, tri;
        double area2;
        if (convex_ok) {
            const double ic = incircle(a, b, d, c);
            diag = ic > 0 ? 1 : 0;
            if (fabs(ic) <= A.flip_tol) diag ^= 1;
            const float fdg = diag == 0 ? edgef(af, df, qxf, qyf) : edgef(bf, cf, qxf, qyf);
            decided = decided && fabsf(fdg) > m;
            if (decided) {
                tri = diag == 0 ? (fdg < 0 ? 0 : 1) : (fdg > 0 ? 0 : 1);
            } else {
                tri = owner_triangle(a, b, c, d, diag, qx, qy);
                if (tri < 0) return;
            }
            const bool s11 = diag == 1 && tri == 1, s00 = diag == 0 && tri == 0;
            area2 = orient(s11 ? b : a, tri == 0 ? b : d, s00 ? d : c);
        } else {
            double ar[2];
            diag = cell_diagonal(a, b, c, d, ar, A.flip_tol);
            if (diag < 0) return;   // folded: the frame is redone by the resolve kernels
            tri = owner_triangle(a, b, c, d, diag, qx, qy);
            if (tri < 0) return;
            area2 = ar[tri];
        }
        // weights as triangle_weights() computes them, with the vertices selected instead of four copies of the code
        // (the lanes of a warp hold all four (diagonal, triangle) cases): (a, b, d), (a, d, c), (a, b, c), (b, d, c)
        const bool t11 = diag == 1 && tri == 1, t00 = diag == 0 && tri == 0, tr0 = tri == 0;
        const P2 p0 = t11 ? b : a, p2 = t00 ? d : c;
        const P2 eu = tr0 ? b : c, ev = tr0 ? p2 : d;   // edge opposite p0, from its smaller-index end point
        const double ee0 = edge_canon(eu, ev, qx, qy), e0 = tr0 ? ee0 : -ee0;
        const double e1 = -edge_canon(p0, p2, qx, qy);
        const double r = drcp(area2);
        double w[3];
        w[0] = dmul(e0, r);
        w[1] = dmul(e1, r);
        w[2] = dsub(dsub(1.0, w[0]), w[1]);
        int k[3];
        k[0] = t11 ? 1 : 0;
        k[1] = tr0 ? 1 : 3;
        k[2] = t00 ? 3 : 2;
        const int v0 = sb + (k[0] >> 1) * SW + (k[0] & 1), v1 = sb + (k[1] >> 1) * SW + (k[1] & 1),
                  v2 = sb + (k[2] >> 1) * SW + (k[2] & 1);
        const size_t px = frame + (size_t)y * A.W + x;
        const bool m0 = s_pm[v0] != 0, m1 = s_pm[v1] != 0, m2 = s_pm[v2] != 0;
        if (CT >= 0) {
            interp_store(s_pay + v0 * PC, s_pay + v1 * PC, s_pay + v2 * PC, m0, m1, m2, w[0], w[1], w[2], PC,
                         A.out + px * PC, A.out_mask ? A.out_mask + px : nullptr, A.rule_strict);
        } else {
            const int il = sb / SW, jc = sb - il * SW;
            const size_t ga = frame + (size_t)(i0 + il) * A.W + j0 + jc;
            const size_t g0 = ga + (size_t)(k[0] >> 1) * A.W + (k[0] & 1), g1 = ga + (size_t)(k[1] >> 1) * A.W + (k[1] & 1),
                         g2 = ga + (size_t)(k[2] >> 1) * A.W + (k[2] & 1);
            interp_store(A.payload + g0 * A.C, A.payload + g1 * A.C, A.payload + g2 * A.C, m0, m1, m2, w[0], w[1], w[2],
                         A.C, A.out + px * A.C, A.out_mask ? A.out_mask + px : nullptr, A.rule_strict);
        }
        if (A.out_mask == nullptr) A.cover[px] = 1;
    };

    // ---------------------------------------------------------------- phase 1: cells -> candidates
    const bool col_ok = gj < A.W - 1;
    int il = ilbase;
    float2 af = s_posf[il * SW + jl], bf = s_posf[il * SW + jl + 1];
    bool vab = s_pt[il * SW + jl] && s_pt[il * SW + jl + 1];
    for (int kr = 0; kr < TH / 4; ++kr, ++il) {
        const int sb = il * SW + jl;
        const float2 cf = s_posf[sb + SW], df = s_posf[sb + SW + 1];
        const bool vcd = s_pt[sb + SW] && s_pt[sb + SW + 1];
        int ncand = 0, x0 = 0, y0 = 0, nx = 1;
        unsigned flag = 0;
        if (col_ok && i0 + il < A.H - 1 && vab && vcd) {
            float xlo = fminf(fminf(af.x, bf.x), fminf(cf.x, df.x)), xhi = fmaxf(fmaxf(af.x, bf.x), fmaxf(cf.x, df.x));
            float ylo = fminf(fminf(af.y, bf.y), fminf(cf.y, df.y)), yhi = fmaxf(fmaxf(af.y, bf.y), fmaxf(cf.y, df.y));
            const float mag = fmaxf(fmaxf(fabsf(xlo), fabsf(xhi)), fmaxf(fabsf(ylo), fabsf(yhi)));
            const float eps = mag * 2.4e-7f + 1e-6f;        // the float32 positions are within half an ulp
            const float ext = (xhi - xlo) + (yhi - ylo) + 1.0f;
            xlo = fmaxf(xlo - eps, lxmin - 1.0f);
            xhi = fminf(xhi + eps, lxmax + 1.0f);
            ylo = fmaxf(ylo - eps, lymin - 1.0f);
            yhi = fminf(yhi + eps, lymax + 1.0f);
            if (xlo <= xhi && ylo <= yhi) {
                x0 = max(ceil_magic(xlo), 0 - ox);
                y0 = max(ceil_magic(ylo), 0 - oy);
                const int x1 = min(floor_magic(xhi), A.W - 1 - ox), y1 = min(floor_magic(yhi), A.H - 1 - oy);
                nx = x1 - x0 + 1;
                const int ny = y1 - y0 + 1;
                if (nx > 0 && ny > 0) ncand = nx * ny;
            }
            if (ncand > 0) {
                const float mo = 16.0f * eps * ext;
                const bool ok = orientf(af, bf, df) > mo && orientf(af, df, cf) > mo && orientf(af, bf, cf) > mo &&
                                orientf(bf, df, cf) > mo;
                if (ok) {
                    flag = REC_OK;
                } else {
                    const P2 a = s_pos[sb], b = s_pos[sb + 1], c = s_pos[sb + SW], d = s_pos[sb + SW + 1];
                    double ar[2];
                    if (cell_diagonal(a, b, c, d, ar, A.flip_tol) < 0) {
                        A.folded[n] = 1;
                        ncand = 0;
                    }
                }
            }
            if (ncand > 4) {   // a stretched cell: rasterised on the spot by the generic float64 loop
                const P2 a = s_pos[sb], b = s_pos[sb + 1], c = s_pos[sb + SW], d = s_pos[sb + SW + 1];
                double ar[2];
                const int diag = cell_diagonal(a, b, c, d, ar, A.flip_tol);
                if (diag >= 0) {
                    EmitDev<CT> e{A, s_pay, s_pm, sb, frame, i0 + il, gj};
                    raster_cell(a, b, c, d, diag, ar, A.W, A.H, e);
                }
                ncand = 0;
            }
        }
        // push: slot s of every cell that has one, compacted over the warp
        int most = ncand;
        for (int o = 16; o > 0; o >>= 1) most = max(most, __shfl_xor_sync(0xffffffffu, most, o));
        for (int sl = 0; sl < most; ++sl) {
            const bool act = sl < ncand;
            const unsigned bal = __ballot_sync(0xffffffffu, act);
            if (act) {
                const int dy = (sl >= nx) + (sl >= 2 * nx) + (sl >= 3 * nx), dx = sl - dy * nx;
                const unsigned rank = __popc(bal & ((1u << lane) - 1u));
                q[(tail + rank) & (QCAP - 1)] =
                    make_uint2((unsigned)sb | flag, (unsigned)(x0 + dx + ox) | ((unsigned)(y0 + dy + oy) << 16));
            }
            tail += __popc(bal);
        }
        __syncwarp();
        while (tail - head >= 32u) drain(32u);
        __syncwarp();
        af = cf;
        bf = df;
        vab = vcd;
    }
    if (tail != head) drain(tail - head);
}

// ------------------------------------------------------------------------------------------- boundary sites -> bins
struct IrrArgs {
    const float* flow;
    const uint8_t* point_mask;
    const int* folded;
    uint32_t* bins;      // [N][nb + 1]
    unsigned long long* occ;   // [N][nc] occupancy words
    uint32_t* sites;     // [N][H * W]
    float sign;
    int H, W, nbx, nby, ncx, ncy;
    int perimeter_only;  // no point mask at all: every frame's boundary sites are the frame border
    const int* masked;   // [N] set when the frame's point mask removes a point; a frame without removed points is
                         // handled like one without a point mask (Flow.apply passes the flow's mask, mostly all true)
    int* isolated;       // [N] set when a valid point of a masked frame has no intact cell around it
    unsigned long long* holes;   // removed points (frame << 32 | index), the candidates for hole_fill()
    unsigned int* hole_count;
    unsigned int hole_cap;
};

__device__ __forceinline__ bool frame_is_plain(const int* masked, int n, int H, int W) {
    return H >= 3 && W >= 3 && (masked == nullptr || masked[n] == 0);
}

__device__ __forceinline__ bool irr_site_of_thread(const IrrArgs& A, int n, long long t, int& row, int& col) {
    if (A.perimeter_only || frame_is_plain(A.masked, n, A.H, A.W)) {
        const long long P = 2ll * A.W + 2ll * (A.H - 2);
        if (t >= P) return false;
        if (t < A.W) {
            row = 0;
            col = (int)t;
        } else if (t < 2ll * A.W) {
            row = A.H - 1;
            col = (int)(t - A.W);
        } else {
            const long long u = t - 2ll * A.W;
            row = 1 + (int)(u >> 1);
            col = (u & 1) ? A.W - 1 : 0;
        }
        return true;
    }
    if (t >= (long long)A.H * A.W) return false;
    row = (int)(t / A.W);
    col = (int)(t - (long long)row * A.W);
    return is_boundary_site(A.point_mask ? A.point_mask + (size_t)n * A.H * A.W : nullptr, A.H, A.W, row, col);
}

// does the point mask of a frame remove anything, and which is its first valid point (raster order)?
__global__ void __launch_bounds__(256) fwd_scan_mask_kernel(const uint8_t* __restrict__ point_mask, size_t frame_px,
                                                            int* __restrict__ masked,
                                                            unsigned int* __restrict__ first_valid) {
    const int n = blockIdx.y;
    const uint8_t* m = point_mask + (size_t)n * frame_px;
    bool zero = false;
    unsigned int first = 0xffffffffu;
    const size_t words = ((reinterpret_cast<uintptr_t>(m) & 15) == 0) ? frame_px / 16 : 0;
    const uint4* m4 = reinterpret_cast<const uint4*>(m);
    for (size_t k = (size_t)blockIdx.x * 256 + threadIdx.x; k < words; k += (size_t)gridDim.x * 256) {
        const uint4 v = m4[k];
        // a zero byte in any of the four words
        const uint32_t z = ((v.x - 0x01010101u) & ~v.x) | ((v.y - 0x01010101u) & ~v.y) | ((v.z - 0x01010101u) & ~v.z) |
                           ((v.w - 0x01010101u) & ~v.w);
        zero = zero || (z & 0x80808080u) != 0u;
        if (first == 0xffffffffu && (v.x | v.y | v.z | v.w) != 0u) {
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
            for (int q = 0; q < 4 && first == 0xffffffffu; ++q)
                if (w4[q]) first = (unsigned int)(k * 16 + q * 4 + ((__ffs(w4[q]) - 1) >> 3));
        }
    }
    for (size_t k = words * 16 + (size_t)blockIdx.x * 256 + threadIdx.x; k < frame_px; k += (size_t)gridDim.x * 256) {
        zero = zero || m[k] == 0;
        if (m[k] != 0 && (unsigned int)k < first) first = (unsigned int)k;
    }
    for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    if ((threadIdx.x & 31) == 0 && first != 0xffffffffu) atomicMin(first_valid + n, first);
    if (__syncthreads_or(zero ? 1 : 0) && threadIdx.x == 0) masked[n] = 1;
}

template <int PASS>   // 0: count sites per bin, 1: fill the site lists (bins hold the end offsets, counted down)
__global__ void __launch_bounds__(256) irr_sites_kernel(const IrrArgs A) {
    const int n = blockIdx.y;
    if (A.folded[n]) return;
    int row, col;
    const size_t frame = (size_t)n * A.H * A.W;
    const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
    const bool site = irr_site_of_thread(A, n, t, row, col);
    if (PASS == 0 && !A.perimeter_only && !frame_is_plain(A.masked, n, A.H, A.W)) {
        // removed points are queued for the small-face pass: one atomic per warp
        const bool removed = !site && t < (long long)A.H * A.W && A.point_mask != nullptr && !A.point_mask[frame + t];
        const unsigned bal = __ballot_sync(0xffffffffu, removed);
        if (bal) {
            const int lane = threadIdx.x & 31, leader = __ffs(bal) - 1;
            unsigned slot = 0;
            if (lane == leader) slot = atomicAdd(A.hole_count, (unsigned)__popc(bal));
            slot = __shfl_sync(0xffffffffu, slot, leader) + __popc(bal & ((1u << lane) - 1u));
            if (removed && slot < A.hole_cap) A.holes[slot] = ((unsigned long long)n << 32) | (unsigned long long)t;
        }
    }
    if (!site) return;
    if (PASS == 0 && A.point_mask != nullptr && !A.perimeter_only && !frame_is_plain(A.masked, n, A.H, A.W) &&
        site_is_isolated(A.point_mask + frame, A.H, A.W, row, col))
        A.isolated[n] = 1;
    const uint32_t id = (uint32_t)(row * A.W + col);
    const float2 f = __ldg(reinterpret_cast<const float2*>(A.flow) + frame + id);
    const P2 p = displaced(f.x, f.y, row, col, A.sign);
    const int bx = bin_coord(p.x, A.nbx), by = bin_coord(p.y, A.nby);
    const int nb = grid_slots(A.nbx, A.nby);
    uint32_t* bins = A.bins + (size_t)n * (nb + 1);
    const int bi = bin_index(A.nbx, bx, by);
    if (PASS == 0) {
        atomicAdd(bins + bi, 1u);
        atomicOr(A.occ + (size_t)n * A.ncx * A.ncy + (by >> COARSE_SHIFT) * A.ncx + (bx >> COARSE_SHIFT),
                 1ull << ((((by & ((1 << COARSE_SHIFT) - 1)) << COARSE_SHIFT)) | (bx & ((1 << COARSE_SHIFT) - 1))));
    } else {
        const uint32_t slot = atomicSub(bins + bi, 1u) - 1u;
        A.sites[frame + slot] = id;
    }
}

// counts -> inclusive end offsets; bins[nb] = number of sites. Three small launches (chunk sums, scan of the chunk
// sums, scan inside the chunks): a single CTA per frame took 100 us for the 130 k bins of a 1080p frame.
constexpr int SCAN_CHUNK = 2048;   // bins per CTA, 8 per thread

__global__ void __launch_bounds__(256) irr_scan_sums_kernel(const uint32_t* bins_all, int nb, uint32_t* chunk_sums,
                                                            int chunks) {
    const uint32_t* a = bins_all + (size_t)blockIdx.y * (nb + 1);
    const int b0 = blockIdx.x * SCAN_CHUNK + threadIdx.x * 8;
    uint32_t sum = 0;
    for (int k = 0; k < 8; ++k)
        if (b0 + k < nb) sum += a[b0 + k];
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    __shared__ uint32_t part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int k = 0; k < 8; ++k) t += part[k];
        chunk_sums[(size_t)blockIdx.y * chunks + blockIdx.x] = t;
    }
}

__global__ void irr_scan_chunks_kernel(uint32_t* chunk_sums, int chunks) {   // exclusive, in place; one warp per frame
    uint32_t* c = chunk_sums + (size_t)blockIdx.x * chunks;
    uint32_t carry = 0;
    for (int base = 0; base < chunks; base += 32) {
        const int i = base + threadIdx.x;
        const uint32_t v = i < chunks ? c[i] : 0u;
        uint32_t inc = v;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if ((int)threadIdx.x >= o) inc += t;
        }
        if (i < chunks) c[i] = carry + inc - v;
        carry += __shfl_sync(0xffffffffu, inc, 31);
    }
}

__global__ void __launch_bounds__(256) irr_scan_final_kernel(uint32_t* bins_all, int nb, const uint32_t* chunk_sums,
                                                             int chunks) {
    uint32_t* a = bins_all + (size_t)blockIdx.y * (nb + 1);
    const int b0 = blockIdx.x * SCAN_CHUNK + threadIdx.x * 8;
    uint32_t v[8], sum = 0;
    for (int k = 0; k < 8; ++k) {
        v[k] = b0 + k < nb ? a[b0 + k] : 0u;
        sum += v[k];
    }
    uint32_t inc = sum;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __shared__ uint32_t part[8];
    if (lane == 31) part[warp] = inc;
    __syncthreads();
    uint32_t run = chunk_sums[(size_t)blockIdx.y * chunks + blockIdx.x] + inc - sum;
    for (int k = 0; k < warp; ++k) run += part[k];
    for (int k = 0; k < 8; ++k) {
        run += v[k];
        if (b0 + k < nb) a[b0 + k] = run;
    }
    if (blockIdx.x == chunks - 1 && threadIdx.x == 255) a[nb] = run;
}

// ------------------------------------------------------------------------------------------------- hull pre-filter
struct HullWs {   // per frame
    unsigned long long dotkey[HULL_DIRS];
    unsigned long long slackkey[HULL_DIRS];
    uint32_t ext[HULL_DIRS];
};

// order-preserving map double -> uint64 (for atomicMax / atomicMin on floating-point values)
__device__ __forceinline__ unsigned long long order_key(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double order_value(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

struct HullArgs {
    const float* flow;
    const int* folded;
    const uint32_t* bins;
    const uint32_t* sites;
    HullWs* ws;
    HullInfo* info;
    HullDirs dirs;
    float sign;
    int H, W, nb;
};

__device__ __forceinline__ SiteGrid hull_grid(const HullArgs& A, int n) {
    SiteGrid g;
    g.H = A.H;
    g.W = A.W;
    g.nbx = g.nby = g.ncx = g.ncy = 0;
    g.bin_start = nullptr;
    g.occ = nullptr;
    g.sites = A.sites + (size_t)n * A.H * A.W;
    g.flow = A.flow + 2 * (size_t)n * A.H * A.W;
    g.sign = A.sign;
    g.inv_w = grid_inv(A.W);
    return g;
}

constexpr int HULL_ITEMS = 8;   // sites per thread

template <int PASS>   // 0: largest dot product per direction, 1: smallest site id among the maximisers, 2: edge slack
__global__ void __launch_bounds__(256) hull_sites_kernel(const HullArgs A) {
    const int n = blockIdx.y;
    if (A.folded[n]) return;
    const uint32_t total = A.bins[(size_t)n * (A.nb + 1) + A.nb];
    const uint32_t s0 = blockIdx.x * (256 * HULL_ITEMS);
    if (s0 >= total) return;
    const SiteGrid g = hull_grid(A, n);
    HullWs& ws = A.ws[n];
    const HullInfo& info = A.info[n];
    const int lane = threadIdx.x & 31;
    const int count = PASS == 2 ? info.m : HULL_DIRS;
    // every thread folds its sites first, one warp reduction and one atomic per direction at the end (with removed
    // points the rims of all holes are boundary sites: a hundred times more of them than on the frame border)
    unsigned long long acc[HULL_DIRS];
#pragma unroll
    for (int k = 0; k < HULL_DIRS; ++k) acc[k] = PASS == 2 ? ~0ull : 0ull;
    for (int it = 0; it < HULL_ITEMS; ++it) {
        const uint32_t s = s0 + it * 256 + threadIdx.x;
        if (s >= total) break;
        const uint32_t id = g.sites[s];
        const P2 p = site_pos(g, id);
#pragma unroll
        for (int k = 0; k < HULL_DIRS; ++k) {
            if (PASS == 0) {
                const unsigned long long key = order_key(dfma(A.dirs.dx[k], p.x, dmul(A.dirs.dy[k], p.y)));
                acc[k] = key > acc[k] ? key : acc[k];
            } else if (PASS == 1) {
                if (order_key(dfma(A.dirs.dx[k], p.x, dmul(A.dirs.dy[k], p.y))) == ws.dotkey[k]) atomicMin(&ws.ext[k], id);
            } else if (k < count) {
                const unsigned long long key = order_key(hull_edge_orient(info, k, p));
                acc[k] = key < acc[k] ? key : acc[k];
            }
        }
    }
    if (PASS == 1) return;
#pragma unroll
    for (int k = 0; k < HULL_DIRS; ++k) {
        if (PASS == 2 && k >= count) break;
        unsigned long long key = acc[k];
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = PASS == 0 ? (other > key ? other : key) : (other < key ? other : key);
        }
        if (lane == 0) {
            if (PASS == 0) {
                if (key != 0ull) atomicMax(&ws.dotkey[k], key);
            } else {
                atomicMin(&ws.slackkey[k], key);
            }
        }
    }
}

template <int PASS>   // 0: polygon of the extreme sites, slack keys reset; 1: slack keys -> HullInfo
__global__ void hull_frame_kernel(const HullArgs A) {
    const int n = blockIdx.x;
    if (A.folded[n]) return;
    HullWs& ws = A.ws[n];
    HullInfo& info = A.info[n];
    if (PASS == 0) {
        if (threadIdx.x == 0) {
            const SiteGrid g = hull_grid(A, n);
            uint32_t ext[HULL_DIRS];
            for (int k = 0; k < HULL_DIRS; ++k) ext[k] = ws.ext[k];
            hull_polygon(g, ext, info);
        }
        if (threadIdx.x < HULL_DIRS) ws.slackkey[threadIdx.x] = order_key(0.0);
    } else if (threadIdx.x < HULL_DIRS) {
        info.slack[threadIdx.x] = order_value(ws.slackkey[threadIdx.x]);
        if ((int)threadIdx.x < info.m) hull_edge_line(info, threadIdx.x);
    }
}

// ---- exact hull: candidates on / beyond the inner polygon, then gift wrapping (one CTA per frame)
struct OuterArgs {
    const float* flow;
    const int* folded;
    const uint32_t* bins;
    const uint32_t* sites;
    const HullInfo* info;
    P2* opos;              // [N][OUTER_CAP]
    uint32_t* oids;        // [N][OUTER_CAP]
    unsigned int* ocount;  // [N]
    HullPoly* poly;        // [N]
    float sign;
    int H, W, nb;
};

__global__ void __launch_bounds__(256) hull_outer_kernel(const OuterArgs A) {
    const int n = blockIdx.y;
    if (A.folded[n]) return;
    const uint32_t total = A.bins[(size_t)n * (A.nb + 1) + A.nb];
    __shared__ HullInfo s_info;
    {
        const int words = sizeof(HullInfo) / 4;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(A.info + n);
        for (int k = threadIdx.x; k < words; k += 256) reinterpret_cast<uint32_t*>(&s_info)[k] = src[k];
    }
    __syncthreads();
    SiteGrid g;
    g.W = A.W;
    g.H = A.H;
    g.sites = A.sites + (size_t)n * A.H * A.W;
    g.flow = A.flow + 2 * (size_t)n * A.H * A.W;
    g.sign = A.sign;
    g.inv_w = grid_inv(A.W);
    for (uint32_t s = blockIdx.x * 256 + threadIdx.x; s < total; s += gridDim.x * 256) {
        const uint32_t id = g.sites[s];
        const P2 p = site_pos(g, id);
        if (!hull_outer_candidate(s_info, p)) continue;
        const unsigned slot = atomicAdd(A.ocount + n, 1u);
        if (slot < (unsigned)OUTER_CAP) {
            A.opos[(size_t)n * OUTER_CAP + slot] = p;
            A.oids[(size_t)n * OUTER_CAP + slot] = id;
        }
    }
}

struct WrapCand {
    P2 p;
    uint32_t id;
};

template <class Better>
__device__ __forceinline__ WrapCand wrap_block_reduce(WrapCand c, Better better, WrapCand* s_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o > 0; o >>= 1) {
        WrapCand other;
        other.p.x = __shfl_xor_sync(0xffffffffu, c.p.x, o);
        other.p.y = __shfl_xor_sync(0xffffffffu, c.p.y, o);
        other.id = __shfl_xor_sync(0xffffffffu, c.id, o);
        if (other.id != NO_SITE && (c.id == NO_SITE || better(other, c))) c = other;
    }
    __syncthreads();
    if (lane == 0) s_warp[warp] = c;
    __syncthreads();
    WrapCand r = s_warp[0];
    for (int k = 1; k < 8; ++k) {
        const WrapCand other = s_warp[k];
        if (other.id != NO_SITE && (r.id == NO_SITE || better(other, r))) r = other;
    }
    return r;
}

__global__ void __launch_bounds__(256) hull_wrap_kernel(const OuterArgs A) {
    const int n = blockIdx.x;
    HullPoly& hp = A.poly[n];
    if (threadIdx.x == 0) {
        hp.m = 0;
        hp.ok = 0;
    }
    if (A.folded[n]) return;
    const unsigned cnt = A.ocount[n];
    if (cnt < 3 || cnt > (unsigned)OUTER_CAP) return;
    const P2* pos = A.opos + (size_t)n * OUTER_CAP;
    const uint32_t* ids = A.oids + (size_t)n * OUTER_CAP;
    __shared__ WrapCand s_warp[8];
    WrapCand c;
    c.id = NO_SITE;
    c.p.x = c.p.y = 0.0;
    for (unsigned k = threadIdx.x; k < cnt; k += 256)
        if (wrap_start_better(pos[k], ids[k], c.p, c.id)) {
            c.p = pos[k];
            c.id = ids[k];
        }
    const WrapCand start = wrap_block_reduce(
        c, [](const WrapCand& q, const WrapCand& b) { return wrap_start_better(q.p, q.id, b.p, b.id); }, s_warp);
    WrapCand cur = start;
    int m = 0;
    for (;;) {
        if (m >= HULL_MAX) return;   // hp.ok stays 0: the searches decide
        if (threadIdx.x == 0) {
            hp.x[m] = cur.p.x;
            hp.y[m] = cur.p.y;
            hp.id[m] = cur.id;
        }
        ++m;
        WrapCand best;
        best.id = NO_SITE;
        best.p = cur.p;
        for (unsigned k = threadIdx.x; k < cnt; k += 256)
            if (wrap_better(cur.p, pos[k], ids[k], best.p, best.id)) {
                best.p = pos[k];
                best.id = ids[k];
            }
        const P2 pivot = cur.p;
        best = wrap_block_reduce(
            best, [pivot](const WrapCand& q, const WrapCand& b) { return wrap_better(pivot, q.p, q.id, b.p, b.id); },
            s_warp);
        if (best.id == NO_SITE || best.id == start.id) break;
        cur = best;
    }
    if (threadIdx.x == 0) {
        hp.m = m;
        hp.ok = m >= 3 ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------------- hull pockets
struct PocketArgs {
    const float* payload;
    const float* flow;
    const uint8_t* payload_mask;
    const int* folded;
    const int* masked;       // [N] or nullptr, see IrrArgs
    const uint32_t* chain;   // [N][chain_cap] traced outer boundary of masked frames (irr_trace_kernel)
    const int* chain_n;      // [N] its length, <= 0: none
    const int* hull_pos;     // [N][HULL_MAX] chain index of every hull vertex
    int chain_cap;
    const HullPoly* poly;
    float* out;
    uint8_t* out_mask;
    uint8_t* cover;
    float sign;
    int C, rule_strict, H, W;
};

struct PocketPixel {
    const PocketArgs& A;
    size_t frame;
    uint32_t v0, v1, v2;
    unsigned long long& count;
    __device__ __forceinline__ void operator()(int x, int y, double w0, double w1, double w2) {
        const size_t px = frame + (size_t)y * A.W + x;
        if (A.cover[px] != UNCOVERED) return;   // only what no intact cell produced
        const uint8_t* pm = A.payload_mask ? A.payload_mask + frame : nullptr;
        const float* pay = A.payload + frame * A.C;
        interp_store(pay + (size_t)v0 * A.C, pay + (size_t)v1 * A.C, pay + (size_t)v2 * A.C, pm ? pm[v0] != 0 : true,
                     pm ? pm[v1] != 0 : true, pm ? pm[v2] != 0 : true, w0, w1, w2, A.C, A.out + px * A.C,
                     A.out_mask ? A.out_mask + px : nullptr, A.rule_strict);
        if (A.out_mask == nullptr) A.cover[px] = 1;
        ++count;
    }
};

struct PocketTri {
    const PocketArgs& A;
    size_t frame;
    Coop coop;
    unsigned long long& count;
    __device__ __forceinline__ void operator()(uint32_t ia, uint32_t ib, uint32_t ic, const P2& pa, const P2& pb,
                                               const P2& pc) {
        PocketPixel px{A, frame, ia, ib, ic, count};
        raster_triangle(pa, pb, pc, ia, ib, ic, A.W, A.H, coop, px);
    }
};

struct PocketSegPixel {
    PocketPixel px;
    __device__ __forceinline__ void operator()(int x, int y, double wa, double wb) { px(x, y, wa, wb, 0.0); }
};

struct PocketSeg {
    const PocketArgs& A;
    size_t frame;
    unsigned long long& count;
    __device__ __forceinline__ void operator()(uint32_t ia, uint32_t ib, const P2& pa, const P2& pb, const Coop& co) {
        PocketSegPixel px{PocketPixel{A, frame, ia, ib, ib, count}};
        raster_segment(pa, pb, A.W, A.H, co, px);
    }
};

__device__ __forceinline__ SiteGrid pocket_grid(const PocketArgs& A, size_t frame) {
    SiteGrid g;
    g.H = A.H;
    g.W = A.W;
    g.nbx = g.nby = g.ncx = g.ncy = 0;
    g.bin_start = nullptr;
    g.occ = nullptr;
    g.sites = nullptr;
    g.flow = A.flow + 2 * frame;
    g.sign = A.sign;
    g.inv_w = grid_inv(A.W);
    return g;
}

// ------------------------------------------------------------------------------------------------- small holes
// One thread per removed point: the first removed point of a small face (hole_loop) triangulates it and rasterises
// the triangles; all other threads find a removed point with a smaller index on their walk and stop.
__global__ void __launch_bounds__(128) irr_holes_kernel(const PocketArgs A, const uint8_t* __restrict__ point_mask,
                                                        const unsigned long long* __restrict__ holes,
                                                        const unsigned int* __restrict__ hole_count,
                                                        unsigned int hole_cap) {
    const unsigned count = min(*hole_count, hole_cap);
    const Coop solo{0, 1};
    unsigned long long pixels = 0;
    for (unsigned it = blockIdx.x * 128 + threadIdx.x; it < count; it += gridDim.x * 128) {
        const unsigned long long item = holes[it];
        const int n = (int)(item >> 32);
        if (A.folded[n]) continue;
        const uint32_t id = (uint32_t)(item & 0xffffffffu);
        const size_t frame = (size_t)n * A.H * A.W;
        const SiteGrid g = pocket_grid(A, frame);
        PocketTri tri{A, frame, solo, pixels};
        hole_fill(g, point_mask + frame, (int)(id / (uint32_t)A.W), (int)(id % (uint32_t)A.W), tri);
    }
    for (int o = 16; o > 0; o >>= 1) pixels += __shfl_xor_sync(0xffffffffu, pixels, o);
    if ((threadIdx.x & 31) == 0 && pixels) atomicAdd(&g_stats[0], pixels);
}

// ------------------------------------------------------------------------------------------------- outer boundary
// trace_outer_loop() of forward_irregular.cuh, one warp per masked frame: the walk is serial, but the nine mask bytes
// around the current vertex are fetched by nine lanes at once (one memory round trip per step). Then the chain index
// of every hull vertex, in one more walk (the hull visits the chain in its own order).
struct TraceArgs {
    const uint8_t* point_mask;
    const int* folded;
    const int* masked;
    const int* isolated;
    const unsigned int* first_valid;
    const HullPoly* poly;
    uint32_t* chain;
    int* chain_n;
    int* hull_pos;
    int chain_cap, H, W;
};

__device__ __forceinline__ unsigned neighbourhood(const uint8_t* pm, int H, int W, int r, int c, int lane) {
    bool v = false;
    if (lane < 9) {
        const int rr = r + lane / 3 - 1, cc = c + lane % 3 - 1;
        v = rr >= 0 && cc >= 0 && rr < H && cc < W && pm[(size_t)rr * W + cc] != 0;
    }
    return __ballot_sync(0xffffffffu, v) & 0x1ffu;   // bit 3 * (dr + 1) + (dc + 1)
}
// quadrant q (SE, SW, NW, NE) of the centre intact?
__device__ __forceinline__ bool nb_quadrant(unsigned nb, int q) {
    const unsigned masks[4] = {0x1b0u /* 4 5 7 8 */, 0x0d8u /* 3 4 6 7 */, 0x01bu /* 0 1 3 4 */, 0x036u /* 1 2 4 5 */};
    const unsigned m = masks[q & 3];
    return (nb & m) == m;
}

__global__ void __launch_bounds__(32) irr_trace_kernel(const TraceArgs A) {
    const int n = blockIdx.x, lane = threadIdx.x;
    if (lane == 0) A.chain_n[n] = 0;
    if (A.folded[n] || A.point_mask == nullptr || frame_is_plain(A.masked, n, A.H, A.W) || A.isolated[n]) return;
    const HullPoly& hp = A.poly[n];
    if (!hp.ok || A.H < 3 || A.W < 3) return;
    const unsigned int first = A.first_valid[n];
    if (first >= (unsigned int)A.H * (unsigned int)A.W) return;
    const uint8_t* pm = A.point_mask + (size_t)n * A.H * A.W;
    uint32_t* out = A.chain + (size_t)n * A.chain_cap;
    const int H = A.H, W = A.W;
    const int r0 = (int)(first / (unsigned)W), c0 = (int)(first % (unsigned)W);
    const int dr[4] = {0, 1, 0, -1}, dc[4] = {1, 0, -1, 0};
    unsigned nb = neighbourhood(pm, H, W, r0, c0, lane);
    int k0 = 2, turns = 0;
    while (!nb_quadrant(nb, k0 + 3)) {
        --k0;
        if (++turns > 3) return;
    }
    k0 &= 3;
    int ar = r0, ac = c0, k = k0, cnt = 0;
    for (;;) {
        if (cnt >= A.chain_cap) return;
        const bool q0 = nb_quadrant(nb, 0), q1 = nb_quadrant(nb, 1), q2 = nb_quadrant(nb, 2), q3 = nb_quadrant(nb, 3);
        if ((q0 && q2 && !q1 && !q3) || (q1 && q3 && !q0 && !q2)) return;   // pinched
        if (lane == 0) out[cnt] = (uint32_t)(ar * W + ac);
        ++cnt;
        const int br = ar + dr[k], bc = ac + dc[k];
        nb = neighbourhood(pm, H, W, br, bc, lane);
        int j = k + 1;
        turns = 0;
        while (!nb_quadrant(nb, j + 3)) {
            --j;
            if (++turns > 3) return;
        }
        ar = br;
        ac = bc;
        k = j & 3;
        if (ar == r0 && ac == c0 && k == k0) break;
    }
    if (cnt < 3) return;
    __syncwarp();
    for (int i = lane; i < cnt / 2; i += 32) {   // the walk has the outside on its left: reversed
        const uint32_t t = out[i];
        out[i] = out[cnt - 1 - i];
        out[cnt - 1 - i] = t;
    }
    __syncwarp();
    // hull vertex e sits at chain index hull_pos[e]: the hull runs through the chain in chain order
    int* pos = A.hull_pos + (size_t)n * HULL_MAX;
    bool ok = true;
    if (lane == 0) {
        int t = 0, scanned = 0;
        for (int e = 0; e < hp.m && ok; ++e) {
            const uint32_t id = hp.id[e];
            while (out[t] != id) {
                t = t + 1 == cnt ? 0 : t + 1;
                if (++scanned > 2 * cnt) {
                    ok = false;
                    break;
                }
            }
            pos[e] = t;
        }
        A.chain_n[n] = ok ? cnt : 0;
    }
}

// the boundary chain of frame n for the pocket pass: the frame border, the traced boundary, or none (c.n == 0)
__device__ __forceinline__ Chain frame_chain(const PocketArgs& A, int n) {
    if (frame_is_plain(A.masked, n, A.H, A.W)) return perimeter_chain(A.H, A.W);
    const int cn = A.chain_n != nullptr ? A.chain_n[n] : 0;
    return Chain{A.chain + (size_t)n * A.chain_cap, cn > 0 ? cn : 0, A.H, A.W};
}

// Frames without removed points, first the pixels exactly on the displaced frame border that no cell produced (a
// straight border: every pixel of a column after an integer shift) ...
__global__ void __launch_bounds__(256) irr_border_edges_kernel(const PocketArgs A) {
    const int n = blockIdx.y;
    if (A.folded[n]) return;
    const Chain ch = frame_chain(A, n);
    if (ch.n == 0) return;
    const size_t frame = (size_t)n * A.H * A.W;
    const SiteGrid g = pocket_grid(A, frame);
    unsigned long long pixels = 0;
    PocketSeg seg{A, frame, pixels};
    pocket_border_edges(g, ch, blockIdx.x * 256 + threadIdx.x, ch.n, gridDim.x * 256, seg);
    for (int o = 16; o > 0; o >>= 1) pixels += __shfl_xor_sync(0xffffffffu, pixels, o);
    if ((threadIdx.x & 31) == 0 && pixels) atomicAdd(&g_stats[0], pixels);
}

// ... then the pockets: a CTA per hull edge triangulates the pocket between that edge and the displaced frame border
// (pocket_triangulate) and rasterises its triangles. A warp works on one part of the arc, its lanes sharing the scans
// and the rows; when it splits a part, the longer half goes to a small pool in shared memory that idle warps draw from.
constexpr int POOL_CAP = 16, POOL_MIN_LEN = 24;

constexpr int TRI_CAP = 96;
struct PocketPool {
    int lo[POOL_CAP], hi[POOL_CAP];
    int n, active, lock;
    // triangles found by a warp that is splitting an arc, rasterised by the CTA's idle warps (a quarter of the time of a
    // split went into rasterising its long thin triangle row by row, on the critical path of a sequential recursion)
    int tn;
    uint32_t ta[TRI_CAP], tb[TRI_CAP], tc[TRI_CAP];
};

__device__ __forceinline__ void pool_lock(PocketPool& p) {
    while (atomicCAS(&p.lock, 0, 1) != 0) __nanosleep(20);
    __threadfence_block();
}
__device__ __forceinline__ void pool_unlock(PocketPool& p) {
    __threadfence_block();
    atomicExch(&p.lock, 0);
}

struct PocketShare {
    PocketPool& pool;
    int lane;
    __device__ __forceinline__ bool operator()(int i, int j) const {
        if (j - i < POOL_MIN_LEN) return false;
        int took = 0;
        if (lane == 0 && *(volatile int*)&pool.n < POOL_CAP / 2) {
            pool_lock(pool);
            if (pool.n < POOL_CAP) {
                pool.lo[pool.n] = i;
                pool.hi[pool.n] = j;
                ++pool.n;
                took = 1;
            }
            pool_unlock(pool);
        }
        return __shfl_sync(0xffffffffu, took, 0) != 0;
    }
};

// tri() of pocket_triangulate inside the pockets kernel: queue the triangle for an idle warp, rasterise it on the spot
// only when the queue is full
struct PocketTriDefer {
    PocketTri now;
    PocketPool& pool;
    int lane;
    __device__ __forceinline__ void operator()(uint32_t ia, uint32_t ib, uint32_t ic, const P2& pa, const P2& pb,
                                               const P2& pc) {
        int took = 0;
        if (lane == 0 && *(volatile int*)&pool.tn < TRI_CAP) {
            pool_lock(pool);
            if (pool.tn < TRI_CAP) {
                pool.ta[pool.tn] = ia;
                pool.tb[pool.tn] = ib;
                pool.tc[pool.tn] = ic;
                ++pool.tn;
                took = 1;
            }
            pool_unlock(pool);
        }
        if (__shfl_sync(0xffffffffu, took, 0) == 0) now(ia, ib, ic, pa, pb, pc);
    }
};

__global__ void __launch_bounds__(256) irr_pockets_kernel(const PocketArgs A) {
    const int n = blockIdx.y;
    if (A.folded[n]) return;
    const HullPoly& hp = A.poly[n];
    if (!hp.ok) return;
    const Chain ch = frame_chain(A, n);
    if (ch.n == 0) return;
    const bool traced = ch.v != nullptr;
    const int* hpos = A.hull_pos + (size_t)n * HULL_MAX;
    __shared__ PocketPool pool;
    // sites and positions of the arc under the hull edge at hand (see ChainArcCached); longer arcs (4K frames) keep the
    // head of the arc here and compute the rest on the fly
    constexpr int ARC_CACHE = 2304;
    __shared__ P2 s_arc_pos[ARC_CACHE];
    __shared__ uint32_t s_arc_id[ARC_CACHE];
    const int lane = threadIdx.x & 31;
    const Coop coop{lane, 32};
    const size_t frame = (size_t)n * A.H * A.W;
    const SiteGrid g = pocket_grid(A, frame);
    unsigned long long pixels = 0;
    PocketTri tri_now{A, frame, coop, pixels};
    PocketTriDefer tri{tri_now, pool, lane};
    PocketSeg seg{A, frame, pixels};
    PocketShare share{pool, lane};
    const int m = hp.m, P = ch.n;
    for (int e = blockIdx.x; e < m; e += gridDim.x) {
        const int e1 = e + 1 == m ? 0 : e + 1;
        const int k0 = traced ? hpos[e] : perim_index(A.H, A.W, hp.id[e]);
        const int k1 = traced ? hpos[e1] : perim_index(A.H, A.W, hp.id[e1]);
        if (k0 < 0 || k1 < 0) continue;
        const int len = ((k1 - k0) % P + P) % P;
        if (len < 2) continue;
        __syncthreads();
        const int ncached = min(len + 1, ARC_CACHE);
        for (int t = threadIdx.x; t < ncached; t += 256) {
            const uint32_t id = chain_site(ch, (k0 + t) % P);
            s_arc_id[t] = id;
            s_arc_pos[t] = site_pos(g, id);
        }
        if (threadIdx.x == 0) {
            pool.lo[0] = 0;
            pool.hi[0] = len;
            pool.n = 1;
            pool.tn = 0;
            pool.active = 0;
            pool.lock = 0;
        }
        __syncthreads();
        for (;;) {
            int got = 0, i = 0, j = 0;
            uint32_t ta = 0, tb = 0, tc = 0;
            if (lane == 0) {
                // Idle warps look at the pool without taking its lock (ncu: seven polling warps per CTA spent 40 % of the
                // kernel's instructions on the lock and kept the one working warp waiting for it whenever it wanted to
                // hand over a part); only a warp that sees work, or sees the end, confirms under the lock.
                const int seen_n = *(volatile int*)&pool.n, seen_tn = *(volatile int*)&pool.tn,
                          seen_active = *(volatile int*)&pool.active;
                if (seen_n > 0 || seen_tn > 0 || seen_active == 0) {
                    pool_lock(pool);
                    if (pool.n > 0) {
                        --pool.n;
                        i = pool.lo[pool.n];
                        j = pool.hi[pool.n];
                        ++pool.active;
                        got = 1;
                    } else if (pool.tn > 0) {
                        --pool.tn;
                        i = pool.tn;          // slot: copied out below, still under the lock
                        ta = pool.ta[i];
                        tb = pool.tb[i];
                        tc = pool.tc[i];
                        ++pool.active;
                        got = 2;
                    } else if (pool.active == 0) {
                        got = -1;
                    }
                    pool_unlock(pool);
                }
            }
            got = __shfl_sync(0xffffffffu, got, 0);
            if (got < 0) break;
            if (got == 0) {
                __nanosleep(400);
                continue;
            }
            if (got == 2) {   // a queued triangle
                ta = __shfl_sync(0xffffffffu, ta, 0);
                tb = __shfl_sync(0xffffffffu, tb, 0);
                tc = __shfl_sync(0xffffffffu, tc, 0);
                tri_now(ta, tb, tc, site_pos(g, ta), site_pos(g, tb), site_pos(g, tc));
                __syncwarp();
                if (lane == 0) {
                    pool_lock(pool);
                    --pool.active;
                    pool_unlock(pool);
                }
                continue;
            }
            i = __shfl_sync(0xffffffffu, i, 0);
            j = __shfl_sync(0xffffffffu, j, 0);
            pocket_triangulate(g, ChainArcCached{ch, k0, s_arc_id, s_arc_pos, ncached}, i, j, coop, tri, share);
            __syncwarp();
            if (lane == 0) {
                pool_lock(pool);
                --pool.active;
                pool_unlock(pool);
            }
        }
        __syncthreads();   // the pixels exactly on the hull edge come after the triangles of its pocket
        if (threadIdx.x < 32) pocket_chord(g, ch, k0, k1, coop, seg);
    }
    for (int o = 16; o > 0; o >>= 1) pixels += __shfl_xor_sync(0xffffffffu, pixels, o);
    if (lane == 0 && pixels) atomicAdd(&g_stats[0], pixels);
}

// ------------------------------------------------------------------------------------------------- uncovered pixels
struct SolveArgs {
    const float* payload;
    const float* flow;
    const uint8_t* payload_mask;
    const int* folded;
    const int* masked;               // [N] or nullptr, see IrrArgs
    const uint32_t* bins;
    const unsigned long long* occ;
    const uint32_t* sites;
    const HullInfo* info;
    const HullPoly* poly;
    float* out;
    uint8_t* out_mask;
    const uint8_t* cover;
    unsigned long long* heavy;       // work items of the pocket pass: frame << 40 | 8-pixel block << 8 | pixel bits
    unsigned int* heavy_count;
    unsigned long long* todo;        // pixels that need a search: frame << 32 | pixel
    unsigned int* todo_count;
    unsigned int todo_cap;
    int lonely_ok;                   // the pocket pass ran: a marked pixel among marked pixels is outside
    float sign;
    int C, rule_strict, H, W, nbx, nby, ncx, ncy;
};

constexpr int SOLVE_SPAN = 4096;          // pixels per CTA, 16 per thread
constexpr int THREAD_BUDGET = 320;        // sites one thread looks at per apex search before the pixel goes to a warp

// a located pixel is written; one outside the hull keeps its marker (fwd_finalize_kernel zeroes whatever is left: a
// marker that turned into 0 here would look like a produced pixel to the neighbour test of irr_solve_kernel)
__device__ __forceinline__ void solve_store(const SolveArgs& A, size_t frame, uint32_t p, int st, const uint32_t (&vid)[3],
                                            const double (&w)[3]) {
    if (st != LOC_FOUND) return;
    const size_t px = frame + p;
    const uint8_t* pm = A.payload_mask ? A.payload_mask + frame : nullptr;
    const float* pay = A.payload + frame * A.C;
    interp_store(pay + (size_t)vid[0] * A.C, pay + (size_t)vid[1] * A.C, pay + (size_t)vid[2] * A.C,
                 pm ? pm[vid[0]] != 0 : true, pm ? pm[vid[1]] != 0 : true, pm ? pm[vid[2]] != 0 : true, w[0], w[1],
                 w[2], A.C, A.out + px * A.C, A.out_mask ? A.out_mask + px : nullptr, A.rule_strict);
}

// Whatever still carries the marker after all passes lies outside the convex hull of the points: 0 / invalid
// (utils.py:254-256).
__global__ void __launch_bounds__(256) fwd_finalize_kernel(float* __restrict__ out, int C, uint8_t* __restrict__ out_mask,
                                                           const uint8_t* __restrict__ cover, size_t frame_px,
                                                           const int* __restrict__ folded) {
    const int n = blockIdx.y;
    if (folded[n]) return;
    const size_t frame = (size_t)n * frame_px;
    for (size_t p0 = ((size_t)blockIdx.x * 256 + threadIdx.x) * 16; p0 < frame_px; p0 += (size_t)gridDim.x * 256 * 16) {
        const uint8_t* cv = cover + frame + p0;
        uint32_t wds[4];
        if (p0 + 16 <= frame_px && (reinterpret_cast<uintptr_t>(cv) & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(cv);
            wds[0] = v.x; wds[1] = v.y; wds[2] = v.z; wds[3] = v.w;
        } else {
            for (int k = 0; k < 4; ++k) {
                wds[k] = 0;
                for (int b = 0; b < 4; ++b)
                    if (p0 + 4 * k + b < frame_px) wds[k] |= (uint32_t)cv[4 * k + b] << (8 * b);
            }
        }
        for (int k = 0; k < 4; ++k) {
            uint32_t hit = ((wds[k] & 0x7f7f7f7fu) + 0x01010101u) & wds[k] & 0x80808080u;   // bytes equal to 0xFF
            while (hit) {
                const int b = (__ffs(hit) - 1) >> 3;
                hit &= hit - 1;
                const size_t px = frame + p0 + 4 * k + b;
                for (int c = 0; c < C; ++c) out[px * C + c] = 0.f;
                if (out_mask) out_mask[px] = 0;
            }
        }
    }
}

// A CTA reads the marker bytes of a span of 4096 pixels (16 bytes per thread) and lists the uncovered ones in shared
// memory, then works through the list one pixel per thread (the searches are long and the uncovered pixels scattered:
// with 2 % of the points removed 8 % of the pixels are bridged; pixel-to-lane mapping would leave most lanes idle). A
// search that looks at more than THREAD_BUDGET sites is abandoned: these are the pixels of hull pockets, whose long
// thin triangles have circles that graze hundreds of border points. They are handed, in blocks of 8 neighbouring
// pixels, to irr_heavy_kernel.
__global__ void __launch_bounds__(256) irr_solve_kernel(const SolveArgs A) {
    const int n = blockIdx.y;
    if (A.folded[n]) return;
    __shared__ HullInfo s_hull;
    __shared__ uint32_t s_list[SOLVE_SPAN];
    __shared__ uint32_t s_warp[8];
    const size_t frame_px = (size_t)A.H * A.W, frame = (size_t)n * frame_px;
    const size_t p0 = (size_t)blockIdx.x * SOLVE_SPAN + (size_t)threadIdx.x * 16;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t hits[4] = {0, 0, 0, 0};
    int mine = 0;
    if (p0 < frame_px) {
        const uint8_t* cv = A.cover + frame + p0;
        uint32_t wds[4];
        if (p0 + 16 <= frame_px && (reinterpret_cast<uintptr_t>(cv) & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(cv);
            wds[0] = v.x; wds[1] = v.y; wds[2] = v.z; wds[3] = v.w;
        } else {
            for (int k = 0; k < 4; ++k) {
                wds[k] = 0;
                for (int b = 0; b < 4; ++b)
                    if (p0 + 4 * k + b < frame_px) wds[k] |= (uint32_t)cv[4 * k + b] << (8 * b);
            }
        }
        for (int k = 0; k < 4; ++k) {
            hits[k] = ((wds[k] & 0x7f7f7f7fu) + 0x01010101u) & wds[k] & 0x80808080u;   // bytes equal to 0xFF
            mine += __popc(hits[k]);
        }
    }
    // ordered compaction: exclusive scan of the per-thread counts
    int inc = mine;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = (uint32_t)inc;
    __syncthreads();
    unsigned count = 0, base = (unsigned)(inc - mine);
    for (int k = 0; k < 8; ++k) {
        if (k < warp) base += s_warp[k];
        count += s_warp[k];
    }
    if (count == 0) return;
    for (int k = 0; k < 4; ++k) {
        uint32_t hit = hits[k];
        while (hit) {
            const int b = (__ffs(hit) - 1) >> 3;
            hit &= hit - 1;
            s_list[base++] = (uint32_t)(p0 + 4 * k + b);
        }
    }
    {
        const int words = sizeof(HullInfo) / 4;
        const uint32_t* src = reinterpret_cast<const uint32_t*>(A.info + n);
        for (int k = threadIdx.x; k < words; k += 256) reinterpret_cast<uint32_t*>(&s_hull)[k] = src[k];
    }
    __syncthreads();
    SiteGrid g;
    g.H = A.H;
    g.W = A.W;
    g.nbx = A.nbx;
    g.nby = A.nby;
    g.ncx = A.ncx;
    g.ncy = A.ncy;
    const int nb = grid_slots(A.nbx, A.nby);
    g.bin_start = A.bins + (size_t)n * (nb + 1);
    g.occ = A.occ + (size_t)n * A.ncx * A.ncy;
    g.sites = A.sites + frame;
    g.flow = A.flow + 2 * frame;
    g.sign = A.sign;
    g.inv_w = grid_inv(A.W);
    const HullPoly& poly = A.poly[n];     // read through L1 / L2: only the pixels next to the hull get that far
    unsigned long long tally[4] = {0, 0, 0, 0};
    const bool plain = frame_is_plain(A.masked, n, A.H, A.W) && poly.ok && A.lonely_ok;   // the pockets have been filled
    // ---- sort out the pixels outside the hull (most of what is marked); the others go to a list of the whole batch,
    // so that the searches run on full warps (irr_search_kernel): done here, every thread on the pixel it found, they
    // were 3 lanes in 32 wide
    __shared__ uint32_t s_todo[SOLVE_SPAN];
    __shared__ unsigned s_ntodo, s_base;
    if (threadIdx.x == 0) s_ntodo = 0;
    __syncthreads();
    for (unsigned e = threadIdx.x; e < count; e += 256) {
        const uint32_t p = s_list[e];
        const int y = (int)(p / (uint32_t)A.W), x = (int)(p - (uint32_t)y * (uint32_t)A.W);
        P2 q;
        q.x = x;
        q.y = y;
        // A frame without removed points has been covered completely (cells, pockets, border): what is left inside
        // the hull are single pixels the fill rule gave to nobody, and those have produced pixels around them. A
        // marked pixel among marked pixels is outside -- no test against the hull (hundreds of edges on a border that
        // is straight only up to float32 rounding) for the empty corners a rotation leaves.
        bool lonely = plain;
        if (plain) {
            for (int dy = -1; dy <= 1 && lonely; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const int yy = y + dy, xx = x + dx;
                    if ((dy | dx) != 0 && yy >= 0 && xx >= 0 && yy < A.H && xx < A.W &&
                        A.cover[frame + (size_t)yy * A.W + xx] != UNCOVERED) {
                        lonely = false;
                        break;
                    }
                }
        }
        if (lonely || hull_rejects(s_hull, q) || (poly.ok && !inside_hull(poly, q))) ++tally[3];
        else s_todo[atomicAdd(&s_ntodo, 1u)] = p;
    }
    __syncthreads();
    const unsigned ntodo = s_ntodo;
    if (ntodo > 0) {
        if (threadIdx.x == 0) s_base = atomicAdd(A.todo_count, ntodo);
        __syncthreads();
        const unsigned base_slot = s_base;
        for (unsigned e = threadIdx.x; e < ntodo; e += 256) {
            const uint32_t p = s_todo[e];
            if (base_slot + e < A.todo_cap) {
                A.todo[base_slot + e] = ((unsigned long long)n << 32) | p;
            } else {   // no room in the list: searched here
                const int y = (int)(p / (uint32_t)A.W), x = (int)(p - (uint32_t)y * (uint32_t)A.W);
                P2 q;
                q.x = x;
                q.y = y;
                uint32_t vid[3];
                double w[3];
                const int st = locate(g, q, vid, w, Coop{0, 1}, NO_BUDGET);
                ++tally[st == LOC_FOUND ? 0 : (st == LOC_OUTSIDE ? 1 : 2)];
                solve_store(A, frame, p, st, vid, w);
            }
        }
    }
    for (int k = 0; k < 4; ++k) {   // one atomic per warp: thousands of threads on one counter serialise in L2
        unsigned long long v = tally[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&g_stats[k], v);
    }
}

__device__ __forceinline__ SiteGrid solve_grid(const SolveArgs& A, int n) {
    const size_t frame = (size_t)n * A.H * A.W;
    SiteGrid g;
    g.H = A.H;
    g.W = A.W;
    g.nbx = A.nbx;
    g.nby = A.nby;
    g.ncx = A.ncx;
    g.ncy = A.ncy;
    const int nb = grid_slots(A.nbx, A.nby);
    g.bin_start = A.bins + (size_t)n * (nb + 1);
    g.occ = A.occ + (size_t)n * A.ncx * A.ncy;
    g.sites = A.sites + frame;
    g.flow = A.flow + 2 * frame;
    g.sign = A.sign;
    g.inv_w = grid_inv(A.W);
    return g;
}

// The searches: one listed pixel per thread, warps full. A search that looks at more than THREAD_BUDGET sites is
// abandoned and handed to irr_heavy_kernel (one warp per pixel).
__global__ void __launch_bounds__(128) irr_search_kernel(const SolveArgs A) {
    const unsigned count = min(*A.todo_count, A.todo_cap);
    const unsigned lane = threadIdx.x & 31;
    unsigned long long tally[3] = {0, 0, 0};
    for (unsigned it0 = blockIdx.x * 128 + (threadIdx.x & ~31u); it0 < count; it0 += gridDim.x * 128) {
        const unsigned it = it0 + lane;
        bool heavy = false;
        unsigned long long key = ~0ull - lane;      // unique per lane unless the pixel goes to the pocket pass
        uint32_t p = 0;
        if (it < count) {
            const unsigned long long item = A.todo[it];
            const int n = (int)(item >> 32);
            p = (uint32_t)(item & 0xffffffffu);
            const size_t frame = (size_t)n * A.H * A.W;
            const SiteGrid g = solve_grid(A, n);
            const int y = (int)(p / (uint32_t)A.W), x = (int)(p - (uint32_t)y * (uint32_t)A.W);
            P2 q;
            q.x = x;
            q.y = y;
            uint32_t vid[3];
            double w[3];
            const int st = locate(g, q, vid, w, Coop{0, 1}, THREAD_BUDGET);
            if (st == LOC_HEAVY) {
                heavy = true;
                key = ((unsigned long long)n << 40) | ((unsigned long long)(p >> 3) << 8);
            } else {
                ++tally[st == LOC_FOUND ? 0 : (st == LOC_OUTSIDE ? 1 : 2)];
                solve_store(A, frame, p, st, vid, w);
            }
        }
        // neighbouring pixels of a row (they sit in neighbouring lanes: the lists keep the pixel order) form one work
        // item of the pocket pass, which locates the second from the triangle of the first
        const unsigned group = __match_any_sync(0xffffffffu, key);
        const unsigned bits = __reduce_or_sync(group, heavy ? (1u << (p & 7)) : 0u);
        if (heavy && lane == (unsigned)(__ffs(group) - 1)) {
            const unsigned slot = atomicAdd(A.heavy_count, 1u);
            A.heavy[slot] = key | bits;
        }
    }
    for (int k = 0; k < 3; ++k) {
        unsigned long long v = tally[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && v) atomicAdd(&g_stats[k], v);
    }
}

// The pocket pass: one warp per work item (up to 8 neighbouring pixels of a row), all 32 lanes scanning the bins of
// every search. The first pixel of a block is located from scratch, the others start from the triangle of their left
// neighbour: a walk from the nearest site crosses dozens of the fan triangles that fill a pocket, from the neighbouring
// pixel's triangle one or two. Items are independent of each other and of the order they were queued in.
__global__ void __launch_bounds__(256) irr_heavy_kernel(const SolveArgs A) {
    const unsigned count = *A.heavy_count;
    const int lane = threadIdx.x & 31;
    const unsigned nwarps = gridDim.x * 8, gwarp = blockIdx.x * 8 + (threadIdx.x >> 5);
    unsigned long long tally[5] = {0, 0, 0, 0, 0};
    for (unsigned it = gwarp; it < count; it += nwarps) {
        ++tally[4];
        const unsigned long long item = A.heavy[it];
        const int n = (int)(item >> 40);
        const uint32_t block = (uint32_t)((item >> 8) & 0xffffffffu), bits = (uint32_t)(item & 0xffu);
        const size_t frame = (size_t)n * A.H * A.W;
        SiteGrid g;
        g.H = A.H;
        g.W = A.W;
        g.nbx = A.nbx;
        g.nby = A.nby;
        g.ncx = A.ncx;
        g.ncy = A.ncy;
        const int nb = grid_slots(A.nbx, A.nby);
        g.bin_start = A.bins + (size_t)n * (nb + 1);
        g.occ = A.occ + (size_t)n * A.ncx * A.ncy;
        g.sites = A.sites + frame;
        g.flow = A.flow + 2 * frame;
        g.sign = A.sign;
    g.inv_w = grid_inv(A.W);
        uint32_t hint[3] = {0, 0, 0};
        bool have_hint = false;
        for (int k = 0; k < 8; ++k) {
            if (!((bits >> k) & 1u)) {
                have_hint = false;
                continue;
            }
            const uint32_t p = block * 8 + k;
            const int y = (int)(p / (uint32_t)A.W), x = (int)(p - (uint32_t)y * (uint32_t)A.W);
            P2 q;
            q.x = x;
            q.y = y;
            uint32_t vid[3];
            double w[3];
            const Coop coop{lane, 32};
            const int st = (have_hint && x > 0) ? locate_hinted(g, q, hint, vid, w, coop, NO_BUDGET)
                                                : locate(g, q, vid, w, coop, NO_BUDGET);
            have_hint = st == LOC_FOUND;
            if (have_hint) {
                hint[0] = vid[0];
                hint[1] = vid[1];
                hint[2] = vid[2];
            }
            if (lane == 0) {
                ++tally[st == LOC_FOUND ? 0 : (st == LOC_OUTSIDE ? 1 : 2)];
                ++tally[3];
                solve_store(A, frame, p, st, vid, w);
            }
        }
    }
    if (lane == 0) {
        for (int k = 0; k < 3; ++k)
            if (tally[k]) atomicAdd(&g_stats[k], tally[k]);
        if (tally[3]) atomicAdd(&g_stats[4], tally[3]);
        if (tally[4]) atomicAdd(&g_stats[5], tally[4]);
    }
}

// ------------------------------------------------------------------------------------------------- workspace layout
struct WsLayout {
    size_t sites, cover, heavy, todo, chain, hull_pos, chain_n, first_valid, isolated, todo_count, heavy_count, hole_count, masked, bins, coarse, hullws, hullinfo, folded, state_side, chunks, opos, oids, ocount, poly, total;
    size_t zero_begin, zero_bytes;   // region cleared before every call (bins, coarse, hull keys, folded flags)
    int nbx, nby, ncx, ncy, nb, nc, chain_cap;
};

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

static WsLayout ws_layout(int N, int H, int W) {
    WsLayout L;
    L.nbx = grid_bins(W);
    L.nby = grid_bins(H);
    L.ncx = grid_coarse(L.nbx);
    L.ncy = grid_coarse(L.nby);
    L.nb = grid_slots(L.nbx, L.nby);
    L.nc = L.ncx * L.ncy;
    const size_t px = (size_t)N * H * W;
    size_t o = 0;
    L.sites = o;            // also the triangle-id plane of the legacy resolve (never used at the same time)
    o = align_up(o + px * 4, 256);
    L.cover = o;
    o = align_up(o + px, 256);
    L.heavy = o;            // at most one item per 8 pixels
    o = align_up(o + px + 8, 256);
    L.todo = o;             // the same for the pixels waiting for a search
    o = align_up(o + px + 8, 256);
    L.chain_cap = 4 * (H + W);   // traced outer boundary of a masked frame
    L.chain = o;
    o = align_up(o + (size_t)N * L.chain_cap * 4, 256);
    L.hull_pos = o;
    o = align_up(o + (size_t)N * HULL_MAX * 4, 256);
    L.chain_n = o;
    o = align_up(o + (size_t)N * 4, 256);
    L.first_valid = o;      // set to ~0 before every call
    o = align_up(o + (size_t)N * 4, 256);
    L.hullinfo = o;
    o = align_up(o + (size_t)N * sizeof(HullInfo), 256);
    L.opos = o;
    o = align_up(o + (size_t)N * OUTER_CAP * sizeof(P2), 256);
    L.oids = o;
    o = align_up(o + (size_t)N * OUTER_CAP * 4, 256);
    L.poly = o;
    o = align_up(o + (size_t)N * sizeof(HullPoly), 256);
    L.zero_begin = o;
    L.bins = o;
    o = align_up(o + (size_t)N * (L.nb + 1) * 4, 256);
    L.coarse = o;
    o = align_up(o + (size_t)N * L.nc * 8, 256);
    L.hullws = o;
    o = align_up(o + (size_t)N * sizeof(HullWs), 256);
    L.folded = o;
    o = align_up(o + (size_t)N * 4, 256);
    L.state_side = o;
    o = align_up(o + (size_t)N * 4, 256);
    L.chunks = o;
    o = align_up(o + (size_t)N * ((L.nb + SCAN_CHUNK - 1) / SCAN_CHUNK) * 4, 256);
    L.heavy_count = o;
    o = align_up(o + 4, 256);
    L.hole_count = o;
    o = align_up(o + 4, 256);
    L.todo_count = o;
    o = align_up(o + 4, 256);
    L.masked = o;
    o = align_up(o + (size_t)N * 4, 256);
    L.isolated = o;
    o = align_up(o + (size_t)N * 4, 256);
    L.ocount = o;
    o = align_up(o + (size_t)N * 4, 256);
    L.zero_bytes = o - L.zero_begin;
    L.total = o;
    return L;
}

__global__ void hull_ws_init_kernel(HullWs* ws, int N) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < N * HULL_DIRS) ws[t / HULL_DIRS].ext[t % HULL_DIRS] = NO_SITE;
}

// Frames whose flow is zero below the threshold are not resampled: apply_flow returns the target itself there
// (utils.py:215-216). frame_state: 0 = resample, 1 = folded (set by the raster kernel), 2 = pass through.
// state_side is the copy read by the kernels that run beside the raster kernel (see ofk_forward_s_ex): 0 or 2 only.
__global__ void fwd_mark_inactive_kernel(const int* __restrict__ flow_nonzero, int* __restrict__ frame_state,
                                         int* __restrict__ state_side, int N) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < N && flow_nonzero[n] == 0) frame_state[n] = state_side[n] = 2;
}

__global__ void __launch_bounds__(256) fwd_passthrough_kernel(const float* __restrict__ payload, int C,
                                                              const uint8_t* __restrict__ payload_mask,
                                                              float* __restrict__ out, uint8_t* __restrict__ out_mask,
                                                              size_t frame_px, const int* __restrict__ frame_state) {
    const int n = blockIdx.y;
    if (frame_state[n] != 2) return;
    const size_t base = (size_t)n * frame_px;
    for (size_t p = (size_t)blockIdx.x * 256 + threadIdx.x; p < frame_px; p += (size_t)gridDim.x * 256) {
        for (int c = 0; c < C; ++c) out[(base + p) * C + c] = payload[(base + p) * C + c];
        if (out_mask) out_mask[base + p] = payload_mask ? (payload_mask[base + p] != 0) : 1;
    }
}

unsigned long long stat(int which) {
#if defined(OFK_FWD_INSTR)
    if (which >= 8 && which < 16) {
        unsigned long long c[8];
        if (cudaMemcpyFromSymbol(c, fwd::g_instr, sizeof(c)) != cudaSuccess) cudaGetLastError();
        return c[which - 8];
    }
#endif
    unsigned long long v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (cudaMemcpyFromSymbol(v, g_stats, sizeof(v)) != cudaSuccess) cudaGetLastError();
    return which >= 0 && which < 8 ? v[which] : 0ull;
}

}  // namespace fwdk

unsigned long long forward_s_stat(int which) { return fwdk::stat(which); }
static std::atomic<double> g_flip_tol{0.0};
static std::atomic<int> g_disable{0};   // test hook, see ofk_forward_s_set_disable

// The boundary-site / hull chain does not depend on the raster kernel: it runs beside it on a library-owned side stream
// (forked from and joined back into the caller's stream with events). One per device; the enqueue of a call holds the
// mutex, so that concurrent callers cannot interleave their fork / join records on the shared events.
struct SideStream {
    std::mutex mu;
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    int state = 0;   // 0 = not created yet, 1 = ready, -1 = unavailable
};
static SideStream g_side[64];
static bool overlap_enabled() {
    static std::atomic<int> v{-1};
    if (v.load() < 0) {
        const char* e = getenv("OFK_FWD_OVERLAP");   // test hook: 0 = everything on the caller's stream
        v.store((e != nullptr && e[0] == '0') ? 0 : 1);
    }
    return v.load() == 1;
}
// with the mutex held
static bool side_ready(SideStream& sd) {
    if (sd.state == 0) {
        int lo = 0, hi = 0;
        sd.state = -1;
        if (cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess &&
            cudaStreamCreateWithPriority(&sd.stream, cudaStreamNonBlocking, hi) == cudaSuccess &&
            cudaEventCreateWithFlags(&sd.fork, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&sd.join, cudaEventDisableTiming) == cudaSuccess)
            sd.state = 1;
        else
            cudaGetLastError();
    }
    return sd.state == 1;
}

}  // namespace ofk

using namespace ofk;

extern "C" int ofk_forward_s_set_flip_tol(double tol) {
    OFK_CHECK_ARG(tol >= 0.0, "ofk_forward_s_set_flip_tol: negative tolerance");
    g_flip_tol.store(tol);
    return OFK_OK;
}

extern "C" int ofk_forward_s_set_disable(int passes) {
    OFK_CHECK_ARG(passes >= 0, "ofk_forward_s_set_disable: negative mask");
    g_disable.store(passes);
    return OFK_OK;
}

extern "C" size_t ofk_forward_s_workspace(int N, int H, int W) {
    if (N <= 0 || H <= 0 || W <= 0) return 0;
    return fwdk::ws_layout(N, H, W).total;
}

template <int CT>
static void launch_raster(const fwdk::RasterArgs& A, int N, cudaStream_t st) {
    using namespace fwdk;
    constexpr int PC = CT > 0 ? CT : 0;
    const size_t smem = (size_t)NV * (sizeof(fwd::P2) + 8 + 2) + 4 * (size_t)(NV * PC + ((NV * PC) & 1)) + 8 * QCAP * 8;
    // > 48 KB of dynamic shared memory needs the opt-in (per device)
    cudaFuncSetAttribute(fwd_raster_kernel<CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    cudaFuncSetAttribute(fwd_raster_kernel<CT>, cudaFuncAttributePreferredSharedMemoryCarveout,
                         cudaSharedmemCarveoutMaxShared);
    dim3 grid((A.W - 1 + TW - 1) / TW, (A.H - 1 + TH - 1) / TH, N);
    fwd_raster_kernel<CT><<<grid, 256, smem, st>>>(A);
}

extern "C" int ofk_forward_s(const float* payload, int C, const float* flow, float flow_sign,
                             const uint8_t* payload_mask, const uint8_t* point_mask, float* out, uint8_t* out_mask,
                             int mask_rule, int N, int H, int W, void* ws, size_t ws_bytes, ofk_stream_t stream) {
    return ofk_forward_s_ex(payload, C, flow, flow_sign, payload_mask, point_mask, nullptr, out, out_mask, mask_rule, N,
                            H, W, ws, ws_bytes, stream);
}

extern "C" int ofk_forward_s_ex(const float* payload, int C, const float* flow, float flow_sign,
                                const uint8_t* payload_mask, const uint8_t* point_mask, const int* flow_nonzero,
                                float* out, uint8_t* out_mask, int mask_rule, int N, int H, int W, void* ws,
                                size_t ws_bytes, ofk_stream_t stream) {
    using namespace fwdk;
    OFK_CHECK_ARG(flow != nullptr, "ofk_forward_s: flow is NULL");
    OFK_CHECK_ARG(N >= 0 && H > 0 && W > 0, "ofk_forward_s: bad shape N=%d H=%d W=%d", N, H, W);
    OFK_CHECK_ARG(C >= 0 && (C == 0 || (payload != nullptr && out != nullptr)), "ofk_forward_s: payload/out NULL");
    OFK_CHECK_ARG(C > 0 || out_mask != nullptr, "ofk_forward_s: nothing to compute");
    OFK_CHECK_ARG(flow_sign == 1.0f || flow_sign == -1.0f, "ofk_forward_s: flow_sign must be +1 or -1");
    OFK_CHECK_ARG(mask_rule == OFK_RULE_STRICT || mask_rule == OFK_RULE_GT_HALF,
                  "ofk_forward_s: mask rule must be STRICT or GT_HALF");
    OFK_CHECK_ARG((size_t)H * W < ((size_t)1 << 29), "ofk_forward_s: frame too large for 32-bit triangle ids");
    OFK_CHECK_ARG(H <= 65535 && W <= 65535, "ofk_forward_s: H=%d / W=%d exceed 65535", H, W);
    OFK_CHECK_ARG((reinterpret_cast<uintptr_t>(flow) & 7) == 0, "ofk_forward_s: flow must be 8-byte aligned");
    if (N == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_forward_s: N=%d exceeds 65535", N);
    const WsLayout L = ws_layout(N, H, W);
    OFK_CHECK_ARG(ws != nullptr && ws_bytes >= L.total, "ofk_forward_s: workspace of %zu bytes needed, got %zu", L.total,
                  ws_bytes);
    cudaStream_t st = as_stream(stream);
    unsigned char* base = static_cast<unsigned char*>(ws);
    uint32_t* d_sites = reinterpret_cast<uint32_t*>(base + L.sites);
    uint8_t* d_cover = out_mask != nullptr ? out_mask : reinterpret_cast<uint8_t*>(base + L.cover);
    uint32_t* d_bins = reinterpret_cast<uint32_t*>(base + L.bins);
    unsigned long long* d_coarse = reinterpret_cast<unsigned long long*>(base + L.coarse);
    HullWs* d_hullws = reinterpret_cast<HullWs*>(base + L.hullws);
    fwd::HullInfo* d_info = reinterpret_cast<fwd::HullInfo*>(base + L.hullinfo);
    int* d_folded = reinterpret_cast<int*>(base + L.folded);
    int* d_state_side = reinterpret_cast<int*>(base + L.state_side);
    const size_t px = (size_t)N * H * W;
    const int strict = mask_rule == OFK_RULE_STRICT ? 1 : 0;

    OFK_CUDA(cudaMemsetAsync(base + L.zero_begin, 0, L.zero_bytes, st));
    OFK_CUDA(cudaMemsetAsync(d_cover, UNCOVERED, px, st));
    hull_ws_init_kernel<<<(N * fwd::HULL_DIRS + 255) / 256, 256, 0, st>>>(d_hullws, N);
    OFK_LAUNCHED();
    if (flow_nonzero != nullptr) {
        fwd_mark_inactive_kernel<<<(N + 255) / 256, 256, 0, st>>>(flow_nonzero, d_folded, d_state_side, N);
        OFK_LAUNCHED();
    }

    // ---- fork: the site / hull chain below goes to the side stream (`ss`), the raster kernel stays on `st`
    cudaStream_t ss = st;
    std::unique_lock<std::mutex> side_lock;
    SideStream* side = nullptr;
    {
        int dev = 0;
        if (overlap_enabled() && H > 1 && W > 1 && cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64) {
            side_lock = std::unique_lock<std::mutex>(g_side[dev].mu);
            if (side_ready(g_side[dev])) {
                side = &g_side[dev];
                ss = side->stream;
                OFK_CUDA(cudaEventRecord(side->fork, st));
                OFK_CUDA(cudaStreamWaitEvent(ss, side->fork, 0));
            } else {
                side_lock.unlock();
            }
        }
    }

    // ---- regular part
    if (H > 1 && W > 1) {
        RasterArgs A{payload, flow, payload_mask, point_mask, out, out_mask, d_cover, d_folded, flow_sign, C, strict,
                     H, W, g_flip_tol.load()};
        switch (C) {
            case 0: launch_raster<0>(A, N, st); break;
            case 1: launch_raster<1>(A, N, st); break;
            case 2: launch_raster<2>(A, N, st); break;
            case 3: launch_raster<3>(A, N, st); break;
            case 4: launch_raster<4>(A, N, st); break;
            default: launch_raster<-1>(A, N, st); break;
        }
        OFK_LAUNCHED();
    }

    // ---- irregular part: boundary sites -> bins -> hull filter -> per-pixel point location
    // (up to the join below on the side stream; these kernels see the frame states 0 / 2 only, a frame the raster kernel
    // finds folded is processed like any other here and skipped by everything after the join)
    // the list of removed points shares its buffer with the work items of the pocket pass (used one after the other)
    const unsigned int hole_cap = (unsigned int)std::min<size_t>(((size_t)N * H * W + 8) / 8, 0xffffffffu);
    int* d_masked = point_mask != nullptr ? reinterpret_cast<int*>(base + L.masked) : nullptr;
    unsigned int* d_first = reinterpret_cast<unsigned int*>(base + L.first_valid);
    int* d_isolated = reinterpret_cast<int*>(base + L.isolated);
    if (point_mask != nullptr) {
        OFK_CUDA(cudaMemsetAsync(d_first, 0xFF, sizeof(unsigned int) * (size_t)N, ss));
        fwd_scan_mask_kernel<<<dim3(std::max(1, std::min(64, (sm_count() * 8 + N - 1) / N)), N), 256, 0, ss>>>(
            point_mask, (size_t)H * W, d_masked, d_first);
        OFK_LAUNCHED();
    }
    IrrArgs I{flow, point_mask, d_state_side, d_bins, d_coarse, d_sites, flow_sign, H, W, L.nbx, L.nby, L.ncx, L.ncy,
              (point_mask == nullptr && H >= 3 && W >= 3) ? 1 : 0, d_masked, d_isolated,
              reinterpret_cast<unsigned long long*>(base + L.heavy),
              reinterpret_cast<unsigned int*>(base + L.hole_count), hole_cap};
    const long long cand = I.perimeter_only ? 2ll * W + 2ll * (H - 2) : (long long)H * W;
    dim3 sgrid((unsigned)((cand + 255) / 256), N);
    irr_sites_kernel<0><<<sgrid, 256, 0, ss>>>(I);
    OFK_LAUNCHED();
    const int chunks = (L.nb + SCAN_CHUNK - 1) / SCAN_CHUNK;
    uint32_t* d_chunks = reinterpret_cast<uint32_t*>(base + L.chunks);
    irr_scan_sums_kernel<<<dim3(chunks, N), 256, 0, ss>>>(d_bins, L.nb, d_chunks, chunks);
    OFK_LAUNCHED();
    irr_scan_chunks_kernel<<<N, 32, 0, ss>>>(d_chunks, chunks);
    OFK_LAUNCHED();
    irr_scan_final_kernel<<<dim3(chunks, N), 256, 0, ss>>>(d_bins, L.nb, d_chunks, chunks);
    OFK_LAUNCHED();
    irr_sites_kernel<1><<<sgrid, 256, 0, ss>>>(I);
    OFK_LAUNCHED();

    HullArgs Hh;
    Hh.flow = flow;
    Hh.folded = d_state_side;
    Hh.bins = d_bins;
    Hh.sites = d_sites;
    Hh.ws = d_hullws;
    Hh.info = d_info;
    for (int k = 0; k < fwd::HULL_DIRS; ++k) {
        Hh.dirs.dx[k] = cos(2.0 * M_PI * k / fwd::HULL_DIRS);
        Hh.dirs.dy[k] = sin(2.0 * M_PI * k / fwd::HULL_DIRS);
    }
    Hh.sign = flow_sign;
    Hh.H = H;
    Hh.W = W;
    Hh.nb = L.nb;
    dim3 hgrid((unsigned)((cand + 256 * HULL_ITEMS - 1) / (256 * HULL_ITEMS)), N);
    hull_sites_kernel<0><<<hgrid, 256, 0, ss>>>(Hh);
    OFK_LAUNCHED();
    hull_sites_kernel<1><<<hgrid, 256, 0, ss>>>(Hh);
    OFK_LAUNCHED();
    hull_frame_kernel<0><<<N, 32, 0, ss>>>(Hh);
    OFK_LAUNCHED();
    hull_sites_kernel<2><<<hgrid, 256, 0, ss>>>(Hh);
    OFK_LAUNCHED();
    hull_frame_kernel<1><<<N, 32, 0, ss>>>(Hh);
    OFK_LAUNCHED();

    OuterArgs O{flow, d_state_side, d_bins, d_sites, d_info, reinterpret_cast<fwd::P2*>(base + L.opos),
                reinterpret_cast<uint32_t*>(base + L.oids), reinterpret_cast<unsigned int*>(base + L.ocount),
                reinterpret_cast<fwd::HullPoly*>(base + L.poly), flow_sign, H, W, L.nb};
    hull_outer_kernel<<<dim3((unsigned)std::min<long long>((cand + 255) / 256, 64), N), 256, 0, ss>>>(O);
    OFK_LAUNCHED();
    hull_wrap_kernel<<<N, 256, 0, ss>>>(O);
    OFK_LAUNCHED();

    uint32_t* d_chain = reinterpret_cast<uint32_t*>(base + L.chain);
    int* d_chain_n = reinterpret_cast<int*>(base + L.chain_n);
    int* d_hull_pos = reinterpret_cast<int*>(base + L.hull_pos);
    const int disable = g_disable.load();
    if (point_mask != nullptr && !(disable & 16)) {   // masked frames: the outer boundary of the mask as the chain
        TraceArgs T{point_mask, d_state_side, d_masked, d_isolated, d_first,
                    reinterpret_cast<const fwd::HullPoly*>(base + L.poly), d_chain, d_chain_n, d_hull_pos, L.chain_cap,
                    H, W};
        irr_trace_kernel<<<N, 32, 0, ss>>>(T);
        OFK_LAUNCHED();
    }
    // ---- join
    if (side != nullptr) {
        OFK_CUDA(cudaEventRecord(side->join, ss));
        OFK_CUDA(cudaStreamWaitEvent(st, side->join, 0));
        side_lock.unlock();
    }
    PocketArgs Pk{payload, flow, payload_mask, d_folded, d_masked, d_chain,
                  (point_mask != nullptr && !(disable & 16)) ? d_chain_n : nullptr,
                  d_hull_pos, L.chain_cap, reinterpret_cast<const fwd::HullPoly*>(base + L.poly), out, out_mask, d_cover,
                  flow_sign, C, strict, H, W};
    if (point_mask != nullptr && H >= 3 && W >= 3 && !(disable & 8)) {
        irr_holes_kernel<<<sm_count() * 8, 128, 0, st>>>(Pk, point_mask, I.holes, I.hole_count, hole_cap);
        OFK_LAUNCHED();
    }
    if (H >= 3 && W >= 3 && !(disable & 4)) {   // frames with a boundary chain (per-frame test inside)
        irr_border_edges_kernel<<<dim3(std::min((L.chain_cap + 255) / 256, 8), N), 256, 0, st>>>(Pk);
        OFK_LAUNCHED();
        // a CTA per hull edge while the batch is small (the pockets of a single frame in parallel)
        irr_pockets_kernel<<<dim3(std::max(1, std::min(fwd::HULL_MAX, (sm_count() * 6 + N - 1) / N)), N), 256, 0, st>>>(Pk);
        OFK_LAUNCHED();
    }

    SolveArgs S{payload, flow, payload_mask, d_folded, d_masked, d_bins, d_coarse, d_sites, d_info,
                reinterpret_cast<const fwd::HullPoly*>(base + L.poly), out, out_mask, d_cover,
                reinterpret_cast<unsigned long long*>(base + L.heavy),
                reinterpret_cast<unsigned int*>(base + L.heavy_count),
                reinterpret_cast<unsigned long long*>(base + L.todo), reinterpret_cast<unsigned int*>(base + L.todo_count),
                hole_cap, (disable & 4) ? 0 : 1, flow_sign, C, strict, H, W, L.nbx, L.nby, L.ncx, L.ncy};
    dim3 vgrid((unsigned)(((size_t)H * W + SOLVE_SPAN - 1) / SOLVE_SPAN), N);
    irr_solve_kernel<<<vgrid, 256, 0, st>>>(S);
    OFK_LAUNCHED();
    irr_search_kernel<<<sm_count() * 8, 128, 0, st>>>(S);
    OFK_LAUNCHED();
    irr_heavy_kernel<<<sm_count() * 4, 256, 0, st>>>(S);
    OFK_LAUNCHED();
    {
        const size_t frame_px = (size_t)H * W;
        const int fin_ctas = (int)std::max<size_t>(1, std::min<size_t>((frame_px + 4095) / 4096,
                                                                       (size_t)std::max(8, 4736 / N)));
        fwd_finalize_kernel<<<dim3(fin_ctas, N), 256, 0, st>>>(out, C, out_mask, d_cover, frame_px, d_folded);
        OFK_LAUNCHED();
    }

    if (flow_nonzero != nullptr) {
        fwd_passthrough_kernel<<<dim3(std::max(8, std::min(1184, 4736 / N)), N), 256, 0, st>>>(
            payload, C, payload_mask, out, out_mask, (size_t)H * W, d_folded);
        OFK_LAUNCHED();
    }
    // ---- folding frames: redone by the order-independent resolve (no-ops for all other frames)
    if (H > 1 && W > 1) {
        unsigned int* winner = reinterpret_cast<unsigned int*>(d_sites);
        const int per_frame = std::max(8, std::min(1184, 4736 / N));   // ~ 8 CTAs per SM over the whole batch
        dim3 lgrid(per_frame, N);
        legacy::fwd_clear<<<lgrid, 256, 0, st>>>(winner, (size_t)H * W, d_folded);
        OFK_LAUNCHED();
        legacy::fwd_scatter<<<lgrid, 256, 0, st>>>(flow, flow_sign, point_mask, winner, H, W, d_folded);
        OFK_LAUNCHED();
        const unsigned long long inv_w = ~0ull / (unsigned long long)W + 1ull;   // ceil(2^64 / W), W >= 2
        legacy::fwd_gather<<<lgrid, 256, 0, st>>>(payload, C, flow, flow_sign, payload_mask, winner, out, out_mask,
                                                 mask_rule, H, W, inv_w, d_folded);
        OFK_LAUNCHED();
    }
    return OFK_OK;
}

// ------------------------------------------------------------------------------------------- scattered -> scattered
// Barycentric interpolation of values attached to the displaced grid at arbitrary query points: replaces the direct
// `griddata(grid - A, A||mask, grid - B, 'linear', fill_value=0)` of combine_with mode 2 / ref 't'
// (flow_class.py:1398-1410) and the griddata calls of track_pts (utils.py:603,614). Same mesh as above (cells split
// along their Delaunay diagonal); the containing triangle of a query is found by a fixed-point walk
// p <- q - sign*flow(p) towards the source cell followed by an exact containment search around it.
namespace ofk {
namespace legacy {

__device__ __forceinline__ P2 mesh_vertex(const float2* __restrict__ fl, int W, int row, int col, float sign,
                                          int pos_f32) {
    const float2 f = __ldg(fl + row * W + col);
    P2 p;
    if (pos_f32) {  // the reference builds these coordinates in float32 (in-place adds on a float32 array)
        p.x = static_cast<double>(__fadd_rn(sign * f.x, static_cast<float>(col)));
        p.y = static_cast<double>(__fadd_rn(sign * f.y, static_cast<float>(row)));
    } else {
        p.x = static_cast<double>(col) + static_cast<double>(sign * f.x);
        p.y = static_cast<double>(row) + static_cast<double>(sign * f.y);
    }
    return p;
}

// tests cell (i, j); on success fills the three vertex indices and barycentric weights
__device__ bool locate_in_cell(const float2* __restrict__ fl, int H, int W, float sign, int pos_f32, int i, int j,
                               double qx, double qy, int (&vidx)[3], double (&w)[3], double flip_tol) {
    if (i < 0 || j < 0 || i >= H - 1 || j >= W - 1) return false;
    P2 v[4];
    v[0] = mesh_vertex(fl, W, i, j, sign, pos_f32);
    v[1] = mesh_vertex(fl, W, i, j + 1, sign, pos_f32);
    v[2] = mesh_vertex(fl, W, i + 1, j, sign, pos_f32);
    v[3] = mesh_vertex(fl, W, i + 1, j + 1, sign, pos_f32);
    const int vid[4] = {i * W + j, i * W + j + 1, (i + 1) * W + j, (i + 1) * W + j + 1};
    const int diag = choose_diagonal(v[0], v[1], v[2], v[3], flip_tol);
    for (int tri = 0; tri < 2; ++tri) {
        const int c0 = corner_of(diag, tri, 0), c1 = corner_of(diag, tri, 1), c2 = corner_of(diag, tri, 2);
        const double area2 = orient(v[c0], v[c1], v[c2]);
        if (area2 == 0.0) continue;
        const double sgn = area2 > 0 ? 1.0 : -1.0;
        const double e0 = edge_fn(v[c1], vid[c1], v[c2], vid[c2], qx, qy);
        const double e1 = edge_fn(v[c2], vid[c2], v[c0], vid[c0], qx, qy);
        const double e2 = edge_fn(v[c0], vid[c0], v[c1], vid[c1], qx, qy);
        if (sgn * e0 >= 0.0 && sgn * e1 >= 0.0 && sgn * e2 >= 0.0) {
            vidx[0] = vid[c0];
            vidx[1] = vid[c1];
            vidx[2] = vid[c2];
            w[0] = e0 / area2;
            w[1] = e1 / area2;
            w[2] = 1.0 - w[0] - w[1];
            return true;
        }
    }
    return false;
}

// The triangle of the mesh p + sign * fl[p] that contains the query (qx, qy): a fixed-point walk towards the source
// position, then an exact containment search in the rings of cells around it. On success fills the three vertex indices
// and the barycentric weights.
__device__ __forceinline__ bool mesh_locate(const float2* __restrict__ fl, int H, int W, float mesh_sign, int pos_f32,
                                            double qx, double qy, int (&vidx)[3], double (&w)[3], double flip_tol) {
    // fixed-point walk towards the source position p with p + sign*flow(p) = q (bilinear flow lookup, clamped)
    double px = qx, py = qy;
    for (int it = 0; it < 12; ++it) {
        const double cx = fmin(fmax(px, 0.0), (double)(W - 1)), cy = fmin(fmax(py, 0.0), (double)(H - 1));
        const int j0 = min((int)cx, W - 2 < 0 ? 0 : W - 2), i0 = min((int)cy, H - 2 < 0 ? 0 : H - 2);
        const double a = cx - j0, b = cy - i0;
        const int j1 = min(j0 + 1, W - 1), i1 = min(i0 + 1, H - 1);
        const float2 f00 = __ldg(fl + i0 * W + j0), f01 = __ldg(fl + i0 * W + j1), f10 = __ldg(fl + i1 * W + j0),
                     f11 = __ldg(fl + i1 * W + j1);
        const double u = (1 - b) * ((1 - a) * f00.x + a * f01.x) + b * ((1 - a) * f10.x + a * f11.x);
        const double v = (1 - b) * ((1 - a) * f00.y + a * f01.y) + b * ((1 - a) * f10.y + a * f11.y);
        const double nx = qx - mesh_sign * u, ny = qy - mesh_sign * v;
        const bool done = fabs(nx - px) < 1e-3 && fabs(ny - py) < 1e-3;
        px = nx;
        py = ny;
        if (done) break;
    }
    bool hit = false;
    const int ci = (int)floor(py), cj = (int)floor(px);
    for (int ring = 0; ring <= 2 && !hit; ++ring) {
        for (int di = -ring; di <= ring && !hit; ++di)
            for (int dj = -ring; dj <= ring && !hit; ++dj) {
                if (max(abs(di), abs(dj)) != ring) continue;
                hit = locate_in_cell(fl, H, W, mesh_sign, pos_f32, ci + di, cj + dj, qx, qy, vidx, w, flip_tol);
            }
    }
    return hit;
}

// channel c of the C-channel payload interpolated with the weights of mesh_locate
__device__ __forceinline__ double mesh_interp(const float* __restrict__ pay, int C, const int (&vidx)[3],
                                              const double (&w)[3], int c) {
    return w[0] * (double)__ldg(pay + (size_t)vidx[0] * C + c) +
           w[1] * (double)__ldg(pay + (size_t)vidx[1] * C + c) +
           w[2] * (double)__ldg(pay + (size_t)vidx[2] * C + c);
}

__global__ void __launch_bounds__(128) mesh_sample_kernel(const float* __restrict__ mesh_flow, float mesh_sign,
                                                          int pos_f32, const float* __restrict__ payload, int C,
                                                          const uint8_t* __restrict__ payload_mask,
                                                          const float* __restrict__ query_flow, float query_sign,
                                                          const double* __restrict__ query_pts, int Q,
                                                          float* __restrict__ out, float* __restrict__ out_maskval,
                                                          uint8_t* __restrict__ found, int H, int W,
                                                          const float* __restrict__ sub_from,
                                                          const uint8_t* __restrict__ sub_mask,
                                                          uint8_t* __restrict__ out_mask8, double flip_tol) {
    const int n = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= Q) return;
    const size_t fbase = (size_t)n * H * W;
    const float2* fl = reinterpret_cast<const float2*>(mesh_flow) + fbase;
    double qx, qy;
    if (query_pts != nullptr) {  // (row, col) pairs
        qy = query_pts[((size_t)n * Q + k) * 2];
        qx = query_pts[((size_t)n * Q + k) * 2 + 1];
    } else {                     // one query per pixel: p + query_sign * query_flow[p]
        const int row = k / W, col = k - row * W;
        const float2 f = __ldg(reinterpret_cast<const float2*>(query_flow) + fbase + k);
        if (pos_f32) {
            qx = static_cast<double>(__fadd_rn(query_sign * f.x, static_cast<float>(col)));
            qy = static_cast<double>(__fadd_rn(query_sign * f.y, static_cast<float>(row)));
        } else {
            qx = static_cast<double>(col) + static_cast<double>(query_sign * f.x);
            qy = static_cast<double>(row) + static_cast<double>(query_sign * f.y);
        }
    }
    int vidx[3];
    double w[3];
    const bool hit = mesh_locate(fl, H, W, mesh_sign, pos_f32, qx, qy, vidx, w, flip_tol);
    const size_t o = (size_t)n * Q + k;
    if (found) found[o] = hit ? 1 : 0;
    float vals[4] = {0.f, 0.f, 0.f, 0.f};
    float mval = 0.f;
    if (hit) {
        const float* pay = payload + fbase * C;
        for (int c = 0; c < C; ++c) {
            const double val = mesh_interp(pay, C, vidx, w, c);
            if (sub_from == nullptr) out[o * C + c] = (float)val;
            else vals[c & 3] = (float)val;
        }
        double m = w[0] + w[1] + w[2];
        if (payload_mask) {
            const uint8_t* pm = payload_mask + fbase;
            m = (pm[vidx[0]] ? w[0] : 0.0) + (pm[vidx[1]] ? w[1] : 0.0) + (pm[vidx[2]] ? w[2] : 0.0);
        }
        mval = (float)m;
    } else if (sub_from == nullptr) {
        for (int c = 0; c < C; ++c) out[o * C + c] = 0.f;
    }
    if (out_maskval) out_maskval[o] = mval;
    if (sub_from != nullptr) {
        // combine_with mode 2 / ref 't' (flow_class.py:1410): B - Flow(resampled A, 't', resampled mask > .99)
        for (int c = 0; c < C; ++c) out[o * C + c] = __fsub_rn(sub_from[o * C + c], vals[c & 3]);
        out_mask8[o] = (mval > 0.99f ? 1 : 0) & (sub_mask ? sub_mask[o] : (uint8_t)1);
    }
}

// Flow.track's mesh route for one float64 point (qy, qx) of the frame fn [H,W,2]: the vector at the point is the
// barycentric interpolation of ofk_mesh_sample, rounded to float32 as ofk_mesh_sample stores it, and the result is
// q + (v, u) in float64. Returns false (and leaves the outputs alone) where no triangle contains the point.
__device__ __forceinline__ bool mesh_track_point(const float* __restrict__ fn, int H, int W, float mesh_sign, double qy,
                                                 double qx, double& orow, double& ocol, double flip_tol) {
    int vidx[3];
    double w[3];
    if (!mesh_locate(reinterpret_cast<const float2*>(fn), H, W, mesh_sign, 0, qx, qy, vidx, w, flip_tol)) return false;
    orow = __dadd_rn(qy, (double)(float)mesh_interp(fn, 2, vidx, w, 1));
    ocol = __dadd_rn(qx, (double)(float)mesh_interp(fn, 2, vidx, w, 0));
    return true;
}

// ofk_track's mesh route: Flow.track for ref 't' (mesh p - flow[p]) and for float points on ref 's' with s_exact_mode
// (mesh_sign = 0:
// the undisplaced grid, the same vertex positions as the zero field Flow.track meshes), one thread per point of the
// flat [N*P] index: out = mesh_track_point, (0, 0) where no triangle contains the point (griddata's NaN rows,
// utils.py:616-618), the points themselves in frames whose flow_nonzero is 0.
template <typename PT>
__global__ void __launch_bounds__(128) track_mesh_kernel(const float* __restrict__ flow,
                                                         const uint8_t* __restrict__ mask, float mesh_sign,
                                                         const int* __restrict__ flow_nonzero,
                                                         const PT* __restrict__ pts, int pts_shared, int P,
                                                         void* __restrict__ out, int int_out,
                                                         const uint8_t* __restrict__ status_plane,
                                                         uint8_t* __restrict__ status, int* __restrict__ errors, int H,
                                                         int W, size_t total, double flip_tol) {
    const size_t hw = (size_t)H * W;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (size_t)gridDim.x * blockDim.x) {
        const size_t n = k / (size_t)P;
        const size_t i = pts_shared ? k - n * P : k;
        const PT r = pts[2 * i], c = pts[2 * i + 1];
        const float* fn = flow + n * hw * 2;
        const float2* fl = reinterpret_cast<const float2*>(fn);
        if (flow_nonzero[n] == 0) {
            store_passthrough<PT, double>(out, int_out, k, r, c);
        } else {
            double orow = 0.0, ocol = 0.0;
            mesh_track_point(fn, H, W, mesh_sign, (double)r, (double)c, orow, ocol, flip_tol);
            store_tracked<double>(out, int_out, k, orow, ocol);
        }
        int err = 0;
        if (status != nullptr)
            track_status(r, c, fl, mask ? mask + n * hw : nullptr, status_plane ? status_plane + n * hw : nullptr, H, W,
                         k, status, err);
        if (err) atomicOr(errors + n, err);
    }
}

// Routes of ofk_track_clips: ref 's' with the float64 bilinear of Flow.track, ref 's' with s_exact_mode (the mesh on
// the undisplaced grid), ref 't' (the mesh p - flow[p]).
enum { CLIPS_S_BILINEAR = 0, CLIPS_S_MESH = 1, CLIPS_T_MESH = 2 };

// (y, x) = round half to even of (r, c); true if that pixel is in the frame (NaN and huge values are not).
__device__ __forceinline__ bool rounded_in_frame(double r, double c, int H, int W, int& y, int& x) {
    y = round_to_i32(r);
    x = round_to_i32(c);
    return y >= 0 && y < H && x >= 0 && x < W;
}

// ofk_track_clips: one thread per trajectory of the flat [S*P] index, walking the L frames of its clip in order with the
// step rules of include/oflib_b200.h. A point lost at step j is NaN in out and 0 in alive from frame s*L + j on.
template <int ROUTE, typename PT>
__global__ void __launch_bounds__(128) track_clips_kernel(const float* __restrict__ flow,
                                                          const uint8_t* __restrict__ mask,
                                                          const int* __restrict__ flow_nonzero,
                                                          const PT* __restrict__ pts, int pts_shared, int L, int P,
                                                          const uint8_t* __restrict__ keep, double* __restrict__ out,
                                                          uint8_t* __restrict__ alive, int H, int W, size_t total,
                                                          double flip_tol) {
    const size_t hw = (size_t)H * W;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);   // numpy's NaN
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (size_t)gridDim.x * blockDim.x) {
        const size_t s = k / (size_t)P, i = k - s * P;
        const size_t src = pts_shared ? i : k;
        double qy = (double)pts[2 * src], qx = (double)pts[2 * src + 1];
        bool live = true;
        for (int j = 0; j < L; ++j) {
            const size_t n = s * L + j, o = n * P + i;
            if (live) {
                const float* fn = flow + n * hw * 2;
                const float2* fl = reinterpret_cast<const float2*>(fn);
                const uint8_t* mn = mask ? mask + n * hw : nullptr;
                int y, x;
                live = rounded_in_frame(qy, qx, H, W, y, x);
                if (ROUTE != CLIPS_T_MESH && live)
                    live = valid_source_s_at(fl, mn, H, W, y, x) && (keep == nullptr || keep[n * hw + (size_t)y * W + x]);
                if (live && flow_nonzero[n] != 0) {
                    if constexpr (ROUTE == CLIPS_S_BILINEAR)
                        live = bilinear_track_point(fl, H, W, qy, qx, qy, qx);
                    else
                        live = mesh_track_point(fn, H, W, ROUTE == CLIPS_T_MESH ? -1.0f : 0.0f, qy, qx, qy, qx, flip_tol);
                }
                if (live) live = rounded_in_frame(qy, qx, H, W, y, x);
                if (ROUTE == CLIPS_T_MESH && live)
                    live = valid_target_t_at(fl, mn, H, W, y, x) && (keep == nullptr || keep[n * hw + (size_t)y * W + x]);
            }
            out[2 * o] = live ? qy : nan;
            out[2 * o + 1] = live ? qx : nan;
            alive[o] = live ? 1 : 0;
        }
    }
}

}  // namespace legacy

int launch_track_mesh(const float* flow, const uint8_t* mask, int ref, const int* flow_nonzero, const void* pts,
                      int pts_dtype, int pts_shared, int P, void* out, int int_out, const uint8_t* status_plane,
                      uint8_t* status, int* errors, int N, int H, int W, cudaStream_t st) {
    const size_t total = (size_t)N * P;
    const float mesh_sign = ref == 't' ? -1.0f : 0.0f;
    const size_t blocks = std::min((total + 127) / 128, (size_t)sm_count() * 64);
    const double tol = g_flip_tol.load();
#define OFK_TRACK_MESH(T)                                                                                              \
    legacy::track_mesh_kernel<T><<<(unsigned)blocks, 128, 0, st>>>(flow, mask, mesh_sign, flow_nonzero,               \
                                                                   static_cast<const T*>(pts), pts_shared, P, out,     \
                                                                   int_out, status_plane, status, errors, H, W, total, \
                                                                   tol)
    switch (pts_dtype) {
        case OFK_F32: OFK_TRACK_MESH(float); break;
        case OFK_F64: OFK_TRACK_MESH(double); break;
        case OFK_I32: OFK_TRACK_MESH(int32_t); break;
        default: OFK_TRACK_MESH(int64_t); break;
    }
#undef OFK_TRACK_MESH
    OFK_LAUNCHED();
    return OFK_OK;
}

int launch_track_clips(const float* flow, const uint8_t* mask, int ref, int exact, const int* flow_nonzero,
                       const void* pts, int pts_dtype, int pts_shared, int S, int L, int P, const uint8_t* keep,
                       double* out, uint8_t* alive, int H, int W, cudaStream_t st) {
    const size_t total = (size_t)S * P;
    const size_t blocks = std::min((total + 127) / 128, (size_t)sm_count() * 64);
    const double tol = g_flip_tol.load();
#define OFK_TRACK_CLIPS(R, T)                                                                                          \
    legacy::track_clips_kernel<legacy::R, T><<<(unsigned)blocks, 128, 0, st>>>(                                        \
        flow, mask, flow_nonzero, static_cast<const T*>(pts), pts_shared, L, P, keep, out, alive, H, W, total, tol)
    const bool f32 = pts_dtype == OFK_F32;
    if (ref == 't') {
        if (f32) OFK_TRACK_CLIPS(CLIPS_T_MESH, float); else OFK_TRACK_CLIPS(CLIPS_T_MESH, double);
    } else if (exact) {
        if (f32) OFK_TRACK_CLIPS(CLIPS_S_MESH, float); else OFK_TRACK_CLIPS(CLIPS_S_MESH, double);
    } else {
        if (f32) OFK_TRACK_CLIPS(CLIPS_S_BILINEAR, float); else OFK_TRACK_CLIPS(CLIPS_S_BILINEAR, double);
    }
#undef OFK_TRACK_CLIPS
    OFK_LAUNCHED();
    return OFK_OK;
}

}  // namespace ofk

extern "C" int ofk_mesh_sample(const float* mesh_flow, float mesh_sign, int pos_f32, const float* payload, int C,
                               const uint8_t* payload_mask, const float* query_flow, float query_sign,
                               const double* query_pts, int Q, float* out, float* out_maskval, uint8_t* found, int N,
                               int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(mesh_flow != nullptr, "ofk_mesh_sample: mesh_flow is NULL");
    OFK_CHECK_ARG((query_flow != nullptr) != (query_pts != nullptr),
                  "ofk_mesh_sample: exactly one of query_flow / query_pts must be given");
    OFK_CHECK_ARG(N >= 0 && H > 1 && W > 1 && C >= 0, "ofk_mesh_sample: bad shape N=%d H=%d W=%d C=%d", N, H, W, C);
    OFK_CHECK_ARG(C == 0 || (payload != nullptr && out != nullptr), "ofk_mesh_sample: payload/out NULL");
    OFK_CHECK_ARG((size_t)H * W < ((size_t)1 << 30), "ofk_mesh_sample: frame too large");
    if (query_flow != nullptr) Q = H * W;
    OFK_CHECK_ARG(Q >= 0, "ofk_mesh_sample: negative query count");
    if (N == 0 || Q == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_mesh_sample: N too large");
    dim3 grid((Q + 127) / 128, N);
    ofk::legacy::mesh_sample_kernel<<<grid, 128, 0, ofk::as_stream(stream)>>>(mesh_flow, mesh_sign, pos_f32, payload, C,
                                                                     payload_mask, query_flow, query_sign, query_pts,
                                                                     Q, out, out_maskval, found, H, W, nullptr,
                                                                     nullptr, nullptr, ofk::g_flip_tol.load());
    OFK_LAUNCHED();
    return OFK_OK;
}

// combine_with(mode = 2) for ref 't' in one launch (flow_class.py:1398-1410): A (vectors and mask) is resampled from
// its source positions grid - A to the source positions grid - B of B (float32 coordinates, no point masking,
// fill 0), subtracted from B, and valid where the resampled mask exceeds .99 and B is valid.
extern "C" int ofk_combine2_t(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float* out,
                              uint8_t* out_mask, int N, int H, int W, ofk_stream_t stream) {
    OFK_CHECK_ARG(A && B && out && out_mask, "ofk_combine2_t: NULL operand");
    OFK_CHECK_ARG(N >= 0 && H > 1 && W > 1, "ofk_combine2_t: bad shape N=%d H=%d W=%d", N, H, W);
    OFK_CHECK_ARG((size_t)H * W < ((size_t)1 << 30), "ofk_combine2_t: frame too large");
    if (N == 0) return OFK_OK;
    OFK_CHECK_ARG(N <= 65535, "ofk_combine2_t: N too large");
    const int Q = H * W;
    dim3 grid((Q + 127) / 128, N);
    ofk::legacy::mesh_sample_kernel<<<grid, 128, 0, ofk::as_stream(stream)>>>(A, -1.0f, 1, A, 2, Am, B, -1.0f, nullptr, Q,
                                                                             out, nullptr, nullptr, H, W, B, Bm,
                                                                             out_mask, ofk::g_flip_tol.load());
    OFK_LAUNCHED();
    return OFK_OK;
}
