// Irregular part of the source-referenced resampler (see forward_geom.cuh): point location in the Delaunay
// triangulation of the "boundary sites" -- the valid displaced pixels that have a removed or missing neighbour
// (frame border, rim of a `consider_mask` hole). Pixels that no intact cell produces can only lie in a Delaunay
// triangle spanned by such sites (or outside the convex hull): scipy.interpolate.griddata triangulates the remaining
// points after the masked ones are dropped (utils.py:249-253 of the reference), bridging holes and filling the
// pockets between the displaced border and its hull.
//
// The sites are binned by position (uniform grid of BIN x BIN pixels over the frame, border bins extend to infinity).
// locate() finds the triangle of a query point q without ever building the triangulation:
//   1. a = site nearest to q, b = site nearest to a: (a, b) is a Delaunay edge (nearest-neighbour graph);
//   2. for the directed edge a -> b with q on its left, the Delaunay triangle on that side has the apex c whose
//      circumcircle through a and b contains no other site on the left (empty-circle criterion; candidates are
//      compared with the in-circle determinant, the search is limited to the bins under the current circle cap);
//      no site on the left at all => (a, b) is a hull edge and q is outside the hull;
//   3. q inside (a, b, c) (edges inclusive) => done; otherwise continue across the edge that separates q from the
//      triangle (visibility walk, terminates on Delaunay triangulations).
// Everything is order independent (ties go to the smaller site index), so the arbitrary order of sites inside a bin
// (filled with atomics on the device) does not influence the result.
#pragma once
#include "forward_geom.cuh"

namespace ofk {
namespace fwd {

#if defined(OFK_FWD_INSTR) && defined(__CUDACC__)   // profiling build only (OFK_FWD_INSTR=1 python -m oflibnumpy_b200.build)
__device__ unsigned long long g_instr[8];
#endif
#if defined(OFK_FWD_INSTR) && defined(__CUDA_ARCH__)
#define OFK_COUNT(i) atomicAdd(&g_instr[i], 1ull)
#else
#define OFK_COUNT(i)
#endif

constexpr int BIN_SHIFT = 2;               // fine bins of 4 x 4 pixels
constexpr int BIN = 1 << BIN_SHIFT;
constexpr int COARSE_SHIFT = 3;            // coarse bins of 8 x 8 fine bins (32 x 32 pixels): one occupancy word each
constexpr uint32_t NO_SITE = 0xffffffffu;
constexpr int HULL_DIRS = 32;

struct SiteGrid {
    int H, W;
    int nbx, nby, ncx, ncy;
    const uint32_t* bin_start; // [nbx * nby + 1] offset of each bin in `sites` (the last entry is the site count)
    const unsigned long long* occ;   // [ncx * ncy] bit (ly * 8 + lx) set when fine bin (lx, ly) of the coarse bin holds a
                                     // site: empty bins are skipped without touching the bin table (a search is a chain
                                     // of dependent loads, and under a thin pocket cap most bins are empty)
    const uint32_t* sites;     // site ids (row * W + col), grouped by bin
    const float* flow;         // [H, W, 2] of this frame
    float sign;
    uint32_t inv_w;            // grid_inv(W): index -> (row, col) without an integer division (0: divide)
};

OFK_HD int grid_bins(int extent) { return (extent + BIN - 1) >> BIN_SHIFT; }
OFK_HD int grid_coarse(int nb) { return (nb + (1 << COARSE_SHIFT) - 1) >> COARSE_SHIFT; }
// slots of the bin table and the slot of a fine bin (row-major over the frame)
OFK_HD int grid_slots(int nbx, int nby) { return nbx * nby; }
OFK_HD int bin_index(int nbx, int bx, int by) { return by * nbx + bx; }

// floor(2^32 / W) + 1: (id * inv) >> 32 is floor(id / W) or one more, for every id < 2^32
OFK_HD uint32_t grid_inv(int W) { return W > 1 ? (uint32_t)(0x100000000ull / (unsigned long long)W) + 1u : 0u; }

OFK_HD P2 site_pos(const SiteGrid& g, uint32_t id) {
    int row, col;
    if (g.inv_w != 0u) {   // every search looks at dozens of sites: the division was a sixth of all instructions
        row = (int)(((unsigned long long)id * g.inv_w) >> 32);
        col = (int)id - row * g.W;
        if (col < 0) {
            --row;
            col += g.W;
        }
    } else {
        row = (int)(id / (uint32_t)g.W);
        col = (int)(id - (uint32_t)row * (uint32_t)g.W);
    }
    const float* f = g.flow + 2 * (size_t)id;
    return displaced(f[0], f[1], row, col, g.sign);
}

// bin coordinate of a position; positions beyond the frame fall into the border bins
OFK_HD int bin_coord(double v, int nb) {
    const double b = floor(v * (1.0 / BIN));
    return b <= 0.0 ? 0 : (b >= (double)(nb - 1) ? nb - 1 : (int)b);
}

OFK_HD int ctz64(unsigned long long v) {   // index of the lowest set bit (v != 0)
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)v) - 1;
#else
    return __builtin_ctzll(v);
#endif
}

OFK_HD bool bin_occupied(const SiteGrid& g, int bx, int by) {
    const int cm = (1 << COARSE_SHIFT) - 1;
    const unsigned long long w = g.occ[(by >> COARSE_SHIFT) * g.ncx + (bx >> COARSE_SHIFT)];
    return (w >> (((by & cm) << COARSE_SHIFT) | (bx & cm))) & 1ull;
}

template <class F>
OFK_HD void scan_bin(const SiteGrid& g, int bx, int by, F& f) {
    if (!bin_occupied(g, bx, by)) return;
    const int b = bin_index(g.nbx, bx, by);
    const uint32_t s0 = g.bin_start[b], s1 = g.bin_start[b + 1];
    for (uint32_t s = s0; s < s1; ++s) {
        const uint32_t id = g.sites[s];
        f(id, site_pos(g, id));
    }
}

// all sites of the bins at Chebyshev distance r from (cx, cy)
template <class F>
OFK_HD void scan_ring(const SiteGrid& g, int cx, int cy, int r, F& f) {
    if (r == 0) {
        scan_bin(g, cx, cy, f);
        return;
    }
    const int x0 = cx - r, x1 = cx + r, y0 = cy - r, y1 = cy + r;
    const int xa = x0 < 0 ? 0 : x0, xb = x1 >= g.nbx ? g.nbx - 1 : x1;
    if (y0 >= 0)
        for (int x = xa; x <= xb; ++x) scan_bin(g, x, y0, f);
    if (y1 < g.nby)
        for (int x = xa; x <= xb; ++x) scan_bin(g, x, y1, f);
    const int ya = y0 + 1 < 0 ? 0 : y0 + 1, yb = y1 - 1 >= g.nby ? g.nby - 1 : y1 - 1;
    if (x0 >= 0)
        for (int y = ya; y <= yb; ++y) scan_bin(g, x0, y, f);
    if (x1 < g.nbx)
        for (int y = ya; y <= yb; ++y) scan_bin(g, x1, y, f);
}

// distance from p (inside the scanned block of bins) to the nearest position that is NOT covered by the bins
// [cx-r, cx+r] x [cy-r, cy+r]; infinity (1e300) when the block covers the whole grid
OFK_HD double ring_reach(const SiteGrid& g, const P2& p, int cx, int cy, int r) {
    double reach = 1e300;
    if (cx - r > 0) reach = fmin(reach, p.x - (double)((cx - r) * BIN));
    if (cx + r < g.nbx - 1) reach = fmin(reach, (double)((cx + r + 1) * BIN) - p.x);
    if (cy - r > 0) reach = fmin(reach, p.y - (double)((cy - r) * BIN));
    if (cy + r < g.nby - 1) reach = fmin(reach, (double)((cy + r + 1) * BIN) - p.y);
    return reach;
}

struct NearestScan {
    const SiteGrid& g;
    P2 p;
    uint32_t exclude, best;
    double best_d2;
    OFK_HD void operator()(uint32_t s, const P2& ps) {
        if (s == exclude) return;
        const double dx = dsub(ps.x, p.x), dy = dsub(ps.y, p.y), d2 = dfma(dx, dx, dmul(dy, dy));
        if (d2 < best_d2 || (d2 == best_d2 && s < best)) {
            best_d2 = d2;
            best = s;
        }
    }
};

OFK_HD uint32_t nearest_site(const SiteGrid& g, const P2& p, uint32_t exclude) {
    const int cx = bin_coord(p.x, g.nbx), cy = bin_coord(p.y, g.nby);
    NearestScan sc{g, p, exclude, NO_SITE, 1e300};
    const int rmax = (g.nbx > g.nby ? g.nbx : g.nby);
    for (int r = 0; r <= rmax; ++r) {
        scan_ring(g, cx, cy, r, sc);
        const double reach = ring_reach(g, p, cx, cy, r);
        if (reach >= 1e300) break;
        if (sc.best != NO_SITE && reach > 0 && sc.best_d2 <= reach * reach) break;
    }
    return sc.best;
}

// circumcircle of (pa, pb, pc) as centre / squared radius; ok = false when the three points are so close to collinear
// that the circle is numerically a half plane
struct Circle {
    double ox, oy, r2;
    bool ok;
};
OFK_HD Circle circumcircle(const P2& pa, const P2& pb, const P2& pc) {
    const double bx = pb.x - pa.x, by = pb.y - pa.y, cx = pc.x - pa.x, cy = pc.y - pa.y;
    const double dd = 2.0 * (bx * cy - by * cx);
    const double b2 = bx * bx + by * by, c2 = cx * cx + cy * cy;
    const double ux = (cy * b2 - by * c2) / dd, uy = (bx * c2 - cx * b2) / dd;
    Circle c;
    c.r2 = ux * ux + uy * uy;
    c.ok = (dd != 0.0) && c.r2 < 1e14;
    c.ox = pa.x + ux;
    c.oy = pa.y + uy;
    return c;
}

struct ApexScan {
    const SiteGrid& g;
    P2 pa, pb, pbest;
    uint32_t a, b, best;
    Circle circ;
    int visited;
    OFK_HD void take(uint32_t s, const P2& ps) {
        best = s;
        pbest = ps;
        circ = circumcircle(pa, pb, ps);
    }
    OFK_HD void operator()(uint32_t s, const P2& ps) {
        ++visited;
        OFK_COUNT(3);   // sites looked at (all searches)
        if (s == a || s == b || s == best) return;
        if (!(orient(pa, pb, ps) > 0)) return;
        if (best == NO_SITE) {
            take(s, ps);
            return;
        }
        // s inside the circle of the current apex -> better (co-circular sets: consistently perturbed)
        if (incircle_sign(pa, pb, pbest, ps, a, b, best, s) > 0) take(s, ps);
    }
    // can the block of bins [bx0, bx1] x [by0, by1] hold a site that beats the current apex? (conservative)
    OFK_HD bool may_hold_better(int bx0, int bx1, int by0, int by1) const {
        const double far = 1e12;
        const double X0 = bx0 <= 0 ? -far : (double)(bx0 * BIN), X1 = bx1 >= g.nbx - 1 ? far : (double)((bx1 + 1) * BIN);
        const double Y0 = by0 <= 0 ? -far : (double)(by0 * BIN), Y1 = by1 >= g.nby - 1 ? far : (double)((by1 + 1) * BIN);
        // left of a -> b: the corner furthest to the left decides
        const double ex = pb.x - pa.x, ey = pb.y - pa.y;
        const double qx = (ey > 0 ? X0 : X1) - pa.x, qy = (ex > 0 ? Y1 : Y0) - pa.y;   // maximises ex*qy - ey*qx
        if (!(ex * qy - ey * qx > 0)) return false;
        if (best == NO_SITE || !circ.ok) return true;
        const double dx = circ.ox < X0 ? X0 - circ.ox : (circ.ox > X1 ? circ.ox - X1 : 0.0);
        const double dy = circ.oy < Y0 ? Y0 - circ.oy : (circ.oy > Y1 ? circ.oy - Y1 : 0.0);
        return dx * dx + dy * dy <= circ.r2 * (1.0 + 1e-9) + 1e-9;
    }
};

// bin range [x0, x1] x [y0, y1] covering the part of the circle left of pa -> pb (the cap that can hold a better apex)
OFK_HD void cap_bins(const SiteGrid& g, const P2& pa, const P2& pb, const Circle& c, int& x0, int& x1, int& y0,
                     int& y1) {
    x0 = 0;
    x1 = g.nbx - 1;
    y0 = 0;
    y1 = g.nby - 1;
    if (!c.ok) return;
    double xlo = fmin(pa.x, pb.x), xhi = fmax(pa.x, pb.x), ylo = fmin(pa.y, pb.y), yhi = fmax(pa.y, pb.y);
    const double rr = sqrt(c.r2) * (1.0 + 1e-9) + 1e-9;
    const P2 ex[4] = {{c.ox - rr, c.oy}, {c.ox + rr, c.oy}, {c.ox, c.oy - rr}, {c.ox, c.oy + rr}};
    // an axis extreme of the circle belongs to the cap when it is left of a -> b (a margin keeps it conservative)
    const double margin = -1e-6 * (fabs(pb.x - pa.x) + fabs(pb.y - pa.y)) * rr;
    for (int k = 0; k < 4; ++k) {
        if (orient(pa, pb, ex[k]) >= margin) {
            xlo = fmin(xlo, ex[k].x);
            xhi = fmax(xhi, ex[k].x);
            ylo = fmin(ylo, ex[k].y);
            yhi = fmax(yhi, ex[k].y);
        }
    }
    x0 = bin_coord(xlo, g.nbx);
    x1 = bin_coord(xhi, g.nbx);
    y0 = bin_coord(ylo, g.nby);
    y1 = bin_coord(yhi, g.nby);
}

// A search can be shared by the lanes of a warp (device only): the bins of the cap sweep are dealt out by bin index,
// every lane keeps the best candidate of its share (pruning with its own candidate stays valid: the overall best lies in
// the cap of every other candidate) and the 32 candidates are reduced with the same in-circle comparison.
// n == 1: a single thread does everything (host build; per-thread searches on the device).
struct Coop {
    int lane, n;
};
constexpr uint32_t OVER_BUDGET = 0xfffffffeu;   // apex_site gave up: more than `budget` sites looked at

OFK_HD void coop_reduce(ApexScan& sc, const Coop& coop) {
#if defined(__CUDA_ARCH__)
    if (coop.n == 1) return;
    for (int o = 16; o > 0; o >>= 1) {
        const uint32_t ob = __shfl_xor_sync(0xffffffffu, sc.best, o);
        P2 op;
        op.x = __shfl_xor_sync(0xffffffffu, sc.pbest.x, o);
        op.y = __shfl_xor_sync(0xffffffffu, sc.pbest.y, o);
        if (ob == NO_SITE || ob == sc.best) continue;
        bool take = sc.best == NO_SITE;
        if (!take) take = incircle_sign(sc.pa, sc.pb, sc.pbest, op, sc.a, sc.b, sc.best, ob) > 0;
        if (take) {
            sc.best = ob;
            sc.pbest = op;
        }
    }
    // rounding can make the comparison non-transitive in degenerate configurations: lane 0 has the last word
    sc.best = __shfl_sync(0xffffffffu, sc.best, 0);
    sc.pbest.x = __shfl_sync(0xffffffffu, sc.pbest.x, 0);
    sc.pbest.y = __shfl_sync(0xffffffffu, sc.pbest.y, 0);
#else
    (void)sc;
    (void)coop;
#endif
}

// apex of the Delaunay triangle left of the directed edge a -> b, NO_SITE if there is no site on that side.
// Every site that beats a candidate lies in that candidate's circle cap, and the cap only shrinks: a few rings of bins
// around the edge midpoint give a first candidate (the final one for the small triangles that bridge holes); whatever
// part of its cap they do not cover is swept through the two-level grid, skipping empty coarse bins and bins the
// current cap does not reach (the long thin triangles of hull pockets).
OFK_HD uint32_t apex_site_impl(const SiteGrid& g, uint32_t a, uint32_t b, const P2& pa, const P2& pb,
                               const Coop& coop, int budget, int& visited) {
    ApexScan sc{g, pa, pb, pa, a, b, NO_SITE, {0.0, 0.0, 0.0, false}, 0};
    struct Tally {   // whatever way the search ends, the sites it looked at count against the caller's budget
        int& total;
        const int& mine;
        OFK_HD ~Tally() { total += mine; }
    } tally{visited, sc.visited};
    P2 mid;
    mid.x = 0.5 * (pa.x + pb.x);
    mid.y = 0.5 * (pa.y + pb.y);
    const int cx = bin_coord(mid.x, g.nbx), cy = bin_coord(mid.y, g.nby);
    constexpr int NEAR_RINGS = 2;
    int x0, x1, y0, y1;
    for (int r = 0; r <= NEAR_RINGS; ++r) {
        scan_ring(g, cx, cy, r, sc);
        if (sc.best == NO_SITE) continue;
        cap_bins(g, pa, pb, sc.circ, x0, x1, y0, y1);
        if (x0 >= cx - r && x1 <= cx + r && y0 >= cy - r && y1 <= cy + r) return sc.best;
    }
    const int cs = COARSE_SHIFT, cw = 1 << cs;
    if (coop.n > 1) {
        // a warp shares the search: the coarse bins under the cap of the first candidate (the whole grid without one)
        // are dealt out to the lanes, every lane sweeps its share pruning with its own best candidate, one reduction
        cap_bins(g, pa, pb, sc.circ, x0, x1, y0, y1);
        const int gx0 = x0 >> cs, gx1 = x1 >> cs, gy0 = y0 >> cs, gy1 = y1 >> cs;
        const int gw = gx1 - gx0 + 1, total = gw * (gy1 - gy0 + 1);
        for (int t = coop.lane; t < total; t += coop.n) {
            const int gy = gy0 + t / gw, gx = gx0 + t % gw;
            unsigned long long word = g.occ[gy * g.ncx + gx];
            if (word == 0ull) continue;
            const int fx0 = (gx << cs) > x0 ? (gx << cs) : x0, fx1 = (gx << cs) + cw - 1 < x1 ? (gx << cs) + cw - 1 : x1;
            const int fy0 = (gy << cs) > y0 ? (gy << cs) : y0, fy1 = (gy << cs) + cw - 1 < y1 ? (gy << cs) + cw - 1 : y1;
            if (!sc.may_hold_better(fx0, fx1, fy0, fy1)) continue;
            while (word) {   // the occupied fine bins of this coarse bin
                const int bit = ctz64(word);
                word &= word - 1;
                const int bx = (gx << cs) | (bit & (cw - 1)), by = (gy << cs) | (bit >> cs);
                if (bx < fx0 || bx > fx1 || by < fy0 || by > fy1) continue;
                if (bx >= cx - NEAR_RINGS && bx <= cx + NEAR_RINGS && by >= cy - NEAR_RINGS && by <= cy + NEAR_RINGS)
                    continue;   // already scanned
                if (!sc.may_hold_better(bx, bx, by, by)) continue;
                scan_bin(g, bx, by, sc);
            }
        }
        coop_reduce(sc, coop);
        return sc.best;
    }
    // sweep the rest of the cap through the two-level grid, rings of coarse bins around the midpoint (near to far: a
    // good candidate early shrinks the cap), until the rings cover the cap of the best candidate
    const int ccx = cx >> cs, ccy = cy >> cs;
    const int rcmax = (g.ncx > g.ncy ? g.ncx : g.ncy);
    for (int rc = 0; rc <= rcmax; ++rc) {
        if (sc.visited > budget) return OVER_BUDGET;
        cap_bins(g, pa, pb, sc.circ, x0, x1, y0, y1);   // whole grid while there is no candidate
        const int gx0 = x0 >> cs, gx1 = x1 >> cs, gy0 = y0 >> cs, gy1 = y1 >> cs;
        if (rc > 0 && gx0 > ccx - rc && gx1 < ccx + rc && gy0 > ccy - rc && gy1 < ccy + rc) break;   // covered
        for (int gy = ccy - rc; gy <= ccy + rc; ++gy) {
            if (gy < gy0 || gy > gy1) continue;
            const bool edge_row = (gy == ccy - rc || gy == ccy + rc);
            for (int gx = ccx - rc; gx <= ccx + rc; gx += (edge_row || rc == 0) ? 1 : 2 * rc) {
                if (gx < gx0 || gx > gx1) continue;
                unsigned long long word = g.occ[gy * g.ncx + gx];
                if (word == 0ull) continue;
                const int fx0 = (gx << cs) > x0 ? (gx << cs) : x0, fx1 = (gx << cs) + cw - 1 < x1 ? (gx << cs) + cw - 1 : x1;
                const int fy0 = (gy << cs) > y0 ? (gy << cs) : y0, fy1 = (gy << cs) + cw - 1 < y1 ? (gy << cs) + cw - 1 : y1;
                if (!sc.may_hold_better(fx0, fx1, fy0, fy1)) continue;
                while (word) {   // the occupied fine bins of this coarse bin
                    const int bit = ctz64(word);
                    word &= word - 1;
                    const int bx = (gx << cs) | (bit & (cw - 1)), by = (gy << cs) | (bit >> cs);
                    if (bx < fx0 || bx > fx1 || by < fy0 || by > fy1) continue;
                    if (bx >= cx - NEAR_RINGS && bx <= cx + NEAR_RINGS && by >= cy - NEAR_RINGS && by <= cy + NEAR_RINGS)
                        continue;   // already scanned
                    if (!sc.may_hold_better(bx, bx, by, by)) continue;
                    scan_bin(g, bx, by, sc);
                }
            }
        }
        if (ccx - rc <= 0 && ccy - rc <= 0 && ccx + rc >= g.ncx - 1 && ccy + rc >= g.ncy - 1) break;   // whole grid
    }
    return sc.best;
}

OFK_HD uint32_t apex_site(const SiteGrid& g, uint32_t a, uint32_t b, const P2& pa, const P2& pb, const Coop& coop,
                          int& budget) {   // budget: sites the caller may still look at (decremented)
    int visited = 0;
    const uint32_t c = apex_site_impl(g, a, b, pa, pb, coop, budget, visited);
    if (budget != 0x7fffffff) budget -= visited;
    return (c != OVER_BUDGET && budget < 0) ? OVER_BUDGET : c;
}

constexpr int LOC_FOUND = 0, LOC_OUTSIDE = 1, LOC_FAILED = 2, LOC_HEAVY = 3;
constexpr int NO_BUDGET = 0x7fffffff;
// a safety net against a walk that cycles on rounding, not a budget: the walk from the nearest site crosses every
// triangle between it and q, and in a frame stretched 3x (a 375 x 1242 non-affine zoom) those are more than 512
#ifndef OFK_LOC_MAX_STEPS
#define OFK_LOC_MAX_STEPS 65536
#endif
constexpr int LOC_MAX_STEPS = OFK_LOC_MAX_STEPS;

// The walk: from the Delaunay edge a -> b (q on its left or on its line) to the triangle that contains q.
OFK_HD int locate_walk(const SiteGrid& g, const P2& q, uint32_t a, uint32_t b, P2 pa, P2 pb, uint32_t (&ids)[3],
                       double (&w)[3], const Coop& coop, int budget) {   // budget: sites of the whole walk
    bool flipped = false;
    for (int step = 0; step < LOC_MAX_STEPS; ++step) {
        if (coop.n > 1 && coop.lane == 0) OFK_COUNT(0);   // steps of cooperative walks
        const uint32_t c = apex_site(g, a, b, pa, pb, coop, budget);
        if (c == OVER_BUDGET) return LOC_HEAVY;
        if (c == NO_SITE) {
            if (!flipped && orient(pa, pb, q) == 0) {   // q on the line through a hull edge: look on the other side
                const uint32_t t = a; a = b; b = t;
                const P2 tp = pa; pa = pb; pb = tp;
                flipped = true;
                continue;
            }
            return LOC_OUTSIDE;
        }
        const P2 pc = site_pos(g, c);
        const double o1 = orient(pb, pc, q), o2 = orient(pc, pa, q);
        if (o1 >= 0 && o2 >= 0) {
            const double r = drcp(orient(pa, pb, pc));
            ids[0] = a; ids[1] = b; ids[2] = c;
            w[0] = dmul(o1, r);
            w[1] = dmul(o2, r);
            w[2] = dsub(dsub(1.0, w[0]), w[1]);
            return LOC_FOUND;
        }
        flipped = false;
        if (o1 < 0 && (o2 >= 0 || o1 < o2)) {   // across b -> c: continue with c -> b (q on its left)
            a = c; pa = pc;
        } else {                                // across c -> a: continue with a -> c
            b = c; pb = pc;
        }
    }
    return LOC_FAILED;
}

// Delaunay triangle of the boundary sites that contains q: vertex ids and barycentric weights
OFK_HD int locate(const SiteGrid& g, const P2& q, uint32_t (&ids)[3], double (&w)[3], const Coop& coop = Coop{0, 1},
                  int budget = NO_BUDGET) {
    uint32_t a = nearest_site(g, q, NO_SITE);
    if (a == NO_SITE) return LOC_OUTSIDE;
    P2 pa = site_pos(g, a);
    if (pa.x == q.x && pa.y == q.y) {   // q is a site: its own value (barycentric weights 1, 0, 0)
        ids[0] = ids[1] = ids[2] = a;
        w[0] = 1.0;
        w[1] = w[2] = 0.0;
        return LOC_FOUND;
    }
    uint32_t b = nearest_site(g, pa, a);
    if (b == NO_SITE) return LOC_OUTSIDE;
    P2 pb = site_pos(g, b);
    if (orient(pa, pb, q) < 0) {
        const uint32_t t = a; a = b; b = t;
        const P2 tp = pa; pa = pb; pb = tp;
    }
    return locate_walk(g, q, a, b, pa, pb, ids, w, coop, budget);
}

// The same with a hint: a Delaunay triangle (ids of a previous, nearby query, positively oriented). q inside it costs
// three orientation tests; otherwise the walk starts across the edge that separates q from it. Pocket triangles are
// long fans: a walk from the nearest site crosses dozens of them, from the neighbouring pixel's triangle one or two.
OFK_HD int locate_hinted(const SiteGrid& g, const P2& q, const uint32_t (&hint)[3], uint32_t (&ids)[3],
                         double (&w)[3], const Coop& coop = Coop{0, 1}, int budget = NO_BUDGET) {
    if (hint[0] == hint[1]) return locate(g, q, ids, w, coop, budget);   // the hint is a site hit, not a triangle
    const P2 p0 = site_pos(g, hint[0]), p1 = site_pos(g, hint[1]), p2 = site_pos(g, hint[2]);
    const double o0 = orient(p1, p2, q), o1 = orient(p2, p0, q), o2 = orient(p0, p1, q);
    if (o0 >= 0 && o1 >= 0 && o2 >= 0) {
        const double r = drcp(orient(p0, p1, p2));
        ids[0] = hint[0]; ids[1] = hint[1]; ids[2] = hint[2];
        w[0] = dmul(o0, r);
        w[1] = dmul(o1, r);
        w[2] = dsub(dsub(1.0, w[0]), w[1]);
        return LOC_FOUND;
    }
    // leave through the most violated edge, reversed so that q is on its left
    if (o0 <= o1 && o0 <= o2) return locate_walk(g, q, hint[2], hint[1], p2, p1, ids, w, coop, budget);
    if (o1 <= o2) return locate_walk(g, q, hint[0], hint[2], p0, p2, ids, w, coop, budget);
    return locate_walk(g, q, hint[1], hint[0], p1, p0, ids, w, coop, budget);
}

// ---------------------------------------------------------------------------------------------- hull pre-filter
// Most pixels that no intact cell produces are simply outside the hull (the empty band of a translation, the corners
// left by a rotation). Per frame: the extreme sites in HULL_DIRS directions form a convex polygon inside the hull;
// `slack[i]` is the most negative orient(v_i, v_i+1, site) over all sites, i.e. how far sites reach beyond edge i.
// A pixel further out than that is outside the hull without any search.
struct HullInfo {
    int m;                         // number of polygon vertices (0: no filter)
    int pad_;
    double vx[HULL_DIRS], vy[HULL_DIRS], slack[HULL_DIRS];
    double la[HULL_DIRS], lb[HULL_DIRS], lc[HULL_DIRS];   // edge i rejects q when la * qx + lb * qy + lc < 0
};

// direction k of the pre-filter (the table is computed once on the host and handed to the device, so both builds
// select the same extreme sites)
struct HullDirs {
    double dx[HULL_DIRS], dy[HULL_DIRS];
};

// candidate for the extreme site in direction k: larger dot product wins, ties go to the smaller id
OFK_HD bool hull_better(double dot, uint32_t id, double best_dot, uint32_t best_id) {
    return best_id == NO_SITE || dot > best_dot || (dot == best_dot && id < best_id);
}

// polygon of the distinct extreme sites in direction order (convex, inside the hull)
OFK_HD void hull_polygon(const SiteGrid& g, const uint32_t (&ext)[HULL_DIRS], HullInfo& h) {
    uint32_t ids[HULL_DIRS];
    int m = 0;
    for (int k = 0; k < HULL_DIRS; ++k) {
        if (ext[k] == NO_SITE) continue;
        if (m > 0 && ids[m - 1] == ext[k]) continue;
        ids[m++] = ext[k];
    }
    while (m > 1 && ids[m - 1] == ids[0]) --m;
    if (m < 3) m = 0;
    h.m = m;
    h.pad_ = 0;
    for (int i = 0; i < m; ++i) {
        const P2 p = site_pos(g, ids[i]);
        h.vx[i] = p.x;
        h.vy[i] = p.y;
        h.slack[i] = 0.0;
    }
}

OFK_HD double hull_edge_orient(const HullInfo& h, int i, const P2& p) {
    const int k = i + 1 == h.m ? 0 : i + 1;
    P2 u, v;
    u.x = h.vx[i]; u.y = h.vy[i];
    v.x = h.vx[k]; v.y = h.vy[k];
    return orient(u, v, p);
}

// line form of edge i once its slack is known: orient(v_i, v_i+1, q) < slack_i - tolerance, written as a linear
// function of q (the tolerance covers the rounding of either form)
OFK_HD void hull_edge_line(HullInfo& h, int i) {
    const int k = i + 1 == h.m ? 0 : i + 1;
    const double dx = h.vx[k] - h.vx[i], dy = h.vy[k] - h.vy[i];
    const double scale = fabs(dx) + fabs(dy) + fabs(h.vx[i]) + fabs(h.vy[i]) + 1.0;
    h.la[i] = -dy;
    h.lb[i] = dx;
    h.lc[i] = dy * h.vx[i] - dx * h.vy[i] - h.slack[i] + 1e-8 * scale * scale;
}

OFK_HD bool hull_rejects(const HullInfo& h, const P2& q) {
    for (int i = 0; i < h.m; ++i)
        if (dfma(h.la[i], q.x, dfma(h.lb[i], q.y, h.lc[i])) < 0) return true;
    return false;
}

// serial reference of the per-frame hull kernel (the host build uses it as is; the device kernel computes the same
// maxima / minima with a block reduction)
inline void hull_build_serial(const SiteGrid& g, uint32_t nsites, const HullDirs& dirs, HullInfo& h) {
    uint32_t ext[HULL_DIRS];
    double best[HULL_DIRS];
    for (int k = 0; k < HULL_DIRS; ++k) {
        ext[k] = NO_SITE;
        best[k] = 0.0;
    }
    for (uint32_t s = 0; s < nsites; ++s) {
        const uint32_t id = g.sites[s];
        const P2 p = site_pos(g, id);
        for (int k = 0; k < HULL_DIRS; ++k) {
            const double dot = dfma(dirs.dx[k], p.x, dmul(dirs.dy[k], p.y));
            if (hull_better(dot, id, best[k], ext[k])) {
                best[k] = dot;
                ext[k] = id;
            }
        }
    }
    hull_polygon(g, ext, h);
    for (uint32_t s = 0; s < nsites; ++s) {
        const P2 p = site_pos(g, g.sites[s]);
        for (int i = 0; i < h.m; ++i) h.slack[i] = fmin(h.slack[i], hull_edge_orient(h, i, p));
    }
    for (int i = 0; i < h.m; ++i) hull_edge_line(h, i);
}

// ---------------------------------------------------------------------------------------------- the exact hull
// Pixels outside the convex hull of the sites are 0 / invalid. A search only finds that out when it reaches a hull
// edge and sweeps the whole half plane beyond it for an apex that does not exist -- the most expensive search there
// is, repeated by every pixel of the band just outside the hull. So the hull itself is built once per frame (gift
// wrapping over the few sites on or beyond the inner polygon) and uncovered pixels are tested against it first.
constexpr int HULL_MAX = 1024;        // hull vertices kept per frame; more: no exact test (the searches decide)
constexpr int OUTER_CAP = 65536;      // candidate sites per frame for the wrap; more: no exact test

struct HullPoly {
    int m, ok;
    double x[HULL_MAX], y[HULL_MAX];
    uint32_t id[HULL_MAX];
};

// a site on or beyond an edge of the inner polygon can be a hull vertex, a site strictly inside it cannot
OFK_HD bool hull_outer_candidate(const HullInfo& h, const P2& p) {
    if (h.m == 0) return true;
    for (int i = 0; i < h.m; ++i)
        if (hull_edge_orient(h, i, p) <= 0) return true;
    return false;
}

// start of the wrap: the lexicographically smallest position (always a hull vertex)
OFK_HD bool wrap_start_better(const P2& q, uint32_t qid, const P2& b, uint32_t bid) {
    if (bid == NO_SITE) return true;
    if (q.x != b.x) return q.x < b.x;
    if (q.y != b.y) return q.y < b.y;
    return qid < bid;
}

// gift wrapping with the interior on the left: from pivot p, q is a better next vertex than b when it lies to the
// right of p -> b; among collinear candidates the farthest one wins (hull vertices only, no points inside edges)
OFK_HD bool wrap_better(const P2& p, const P2& q, uint32_t qid, const P2& b, uint32_t bid) {
    if (q.x == p.x && q.y == p.y) return false;
    if (bid == NO_SITE) return true;
    const double o = orient(p, b, q);
    if (o != 0.0) return o < 0;
    const double qx = dsub(q.x, p.x), qy = dsub(q.y, p.y), bx = dsub(b.x, p.x), by = dsub(b.y, p.y);
    const double dq = dfma(qx, qx, dmul(qy, qy)), db = dfma(bx, bx, dmul(by, by));
    // the same direction from p: farther wins. Opposite directions cannot both be candidates of a hull pivot.
    if (dq != db) return dq > db;
    return qid < bid;
}

OFK_HD bool inside_hull(const HullPoly& hp, const P2& q) {
    for (int i = 0; i < hp.m; ++i) {
        const int k = i + 1 == hp.m ? 0 : i + 1;
        P2 u, v;
        u.x = hp.x[i]; u.y = hp.y[i];
        v.x = hp.x[k]; v.y = hp.y[k];
        if (orient(u, v, q) < 0) return false;
    }
    return true;
}

// serial reference of the wrap (host build); pos / ids: the outer candidates
inline void hull_wrap_serial(const P2* pos, const uint32_t* ids, int n, HullPoly& hp) {
    hp.m = 0;
    hp.ok = 0;
    if (n < 3 || n > OUTER_CAP) return;
    int start = -1;
    for (int k = 0; k < n; ++k)
        if (start < 0 || wrap_start_better(pos[k], ids[k], pos[start], ids[start])) start = k;
    int cur = start;
    for (;;) {
        if (hp.m >= HULL_MAX) {
            hp.m = 0;
            return;
        }
        hp.x[hp.m] = pos[cur].x;
        hp.y[hp.m] = pos[cur].y;
        hp.id[hp.m] = ids[cur];
        ++hp.m;
        int best = -1;
        for (int k = 0; k < n; ++k)
            if (wrap_better(pos[cur], pos[k], ids[k], best < 0 ? pos[cur] : pos[best], best < 0 ? NO_SITE : ids[best]))
                best = k;
        if (best < 0 || best == start) break;
        cur = best;
    }
    hp.ok = hp.m >= 3 ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------ hull pockets
// Without removed points the boundary sites are the frame border, a closed chain in a known order, and the region
// between the displaced border and its hull falls into pockets: one per hull edge, bounded by that edge and the arc
// of the chain between its end points. A pocket holds no site, so its Delaunay triangles only have vertices of its own
// arc -- it is triangulated directly, by splitting: the triangle on the base edge (v_i, v_j) has the apex v_k, i < k < j,
// whose circumcircle holds no other vertex of the arc; (v_i, v_k) and (v_k, v_j) are the next base edges. Every
// triangle is found once and rasterised with the fill rule of the regular part, so that the pixels of a pocket (long
// thin fans, the most expensive point locations there are) never reach the per-pixel search.
//
// Border in the orientation of the hull wrap (interior on the left): top row left to right, right column downwards,
// bottom row right to left, left column upwards.
OFK_HD int perim_count(int H, int W) { return 2 * W + 2 * H - 4; }   // H, W >= 2

OFK_HD uint32_t perim_site(int H, int W, int k) {
    if (k < W) return (uint32_t)k;
    k -= W;
    if (k < H - 1) return (uint32_t)((k + 1) * W + W - 1);
    k -= H - 1;
    if (k < W - 1) return (uint32_t)((H - 1) * W + (W - 2 - k));
    k -= W - 1;
    return (uint32_t)((H - 2 - k) * W);
}

OFK_HD int perim_index(int H, int W, uint32_t id) {
    const int row = (int)(id / (uint32_t)W), col = (int)(id - (uint32_t)row * (uint32_t)W);
    if (row == 0) return col;
    if (col == W - 1) return W + row - 1;
    if (row == H - 1) return W + H - 1 + (W - 2 - col);
    if (col == 0) return 2 * W + H - 2 + (H - 2 - row);
    return -1;
}

struct ArcBest {
    uint32_t id;
    int t;
    P2 p;
    double omin, omax, umin, umax;   // range of orient(a, b, .) and of (. - a) . (b - a) over the arc's vertices
};

#if defined(__CUDA_ARCH__)
// warp-wide minimum / maximum of a double as a float rounded outwards (one REDUX on an order-preserving integer key
// instead of five rounds of 64-bit shuffles): for bounds that only have to be conservative
__device__ __forceinline__ int arc_float_key(float f) {
    const int k = __float_as_int(f);
    return k >= 0 ? k : k ^ 0x7fffffff;
}
__device__ __forceinline__ double arc_warp_min(double v) {
    const int k = __reduce_min_sync(0xffffffffu, arc_float_key(__double2float_rd(v)));
    return (double)__int_as_float(k >= 0 ? k : k ^ 0x7fffffff);
}
__device__ __forceinline__ double arc_warp_max(double v) {
    const int k = __reduce_max_sync(0xffffffffu, arc_float_key(__double2float_ru(v)));
    return (double)__int_as_float(k >= 0 ? k : k ^ 0x7fffffff);
}
#endif

OFK_HD void arc_reduce(ArcBest& b, const P2& pa, const P2& pb, uint32_t ia, uint32_t ib, const Coop& coop) {
#if defined(__CUDA_ARCH__)
    if (coop.n == 1) return;
    // the extent of the part (it only feeds the conservative pixel test of pocket_may_hold_pixel) ...
    b.omin = arc_warp_min(b.omin);
    b.omax = arc_warp_max(b.omax);
    b.umin = arc_warp_min(b.umin);
    b.umax = arc_warp_max(b.umax);
    // ... and the apex: exact, a tree of in-circle tests
    for (int o = 16; o > 0; o >>= 1) {
        ArcBest ob;
        ob.id = __shfl_xor_sync(0xffffffffu, b.id, o);
        ob.t = __shfl_xor_sync(0xffffffffu, b.t, o);
        ob.p.x = __shfl_xor_sync(0xffffffffu, b.p.x, o);
        ob.p.y = __shfl_xor_sync(0xffffffffu, b.p.y, o);
        if (ob.id == NO_SITE || ob.id == b.id) continue;
        if (b.id == NO_SITE || incircle_sign(pa, pb, b.p, ob.p, ia, ib, b.id, ob.id) > 0) {
            b.id = ob.id;
            b.t = ob.t;
            b.p = ob.p;
        }
    }
    b.id = __shfl_sync(0xffffffffu, b.id, 0);   // lane 0 has the last word (see coop_reduce)
    b.t = __shfl_sync(0xffffffffu, b.t, 0);
    b.p.x = __shfl_sync(0xffffffffu, b.p.x, 0);
    b.p.y = __shfl_sync(0xffffffffu, b.p.y, 0);
#else
    (void)b; (void)pa; (void)pb; (void)ia; (void)ib; (void)coop;
#endif
}

// Can the part of a pocket over the base edge (pa, pb) hold a pixel? It lies inside the oriented rectangle that bounds
// its vertices: orient(pa, pb, .) in [omin, omax], (. - pa) . (pb - pa) in [umin, umax]. A border that is straight up
// to the rounding of its float32 flow values (every affine field) consists of slivers a few 1e-6 px thick: thousands
// of triangles per frame that contain no pixel and are not worth finding. Conservative: false only if no lattice
// point of the frame lies in the rectangle (widened by a tolerance far above the rounding of this test).
OFK_HD bool pocket_may_hold_pixel(const P2& pa, const P2& pb, const ArcBest& b, int W, int H, const Coop& coop) {
    const double dx = pb.x - pa.x, dy = pb.y - pa.y, len2 = dx * dx + dy * dy;
    if (!(len2 > 0.0)) return true;
    const double len = sqrt(len2);
    const double tol = 1e-7;
    const double a = b.omin / len - tol, c = b.omax / len + tol;        // signed distance from the base line
    if (c - a >= 0.5) return true;
    const double t0 = b.umin / len2, t1 = b.umax / len2;                  // extent along the base edge
    const bool major_x = fabs(dx) >= fabs(dy);
    // extent of the rectangle along the major axis (its corners: pa + t d + s n, n = (-dy, dx) / len)
    const double nx = -dy / len, ny = dx / len;
    double lo = 1e300, hi = -1e300;
    for (int k = 0; k < 4; ++k) {
        const double t = (k & 1) ? t1 : t0, sd = (k & 2) ? c : a;
        const double v = major_x ? pa.x + t * dx + sd * nx : pa.y + t * dy + sd * ny;
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
    const double lim = (double)((major_x ? W : H) - 1);
    if (!(hi >= 0.0 && lo <= lim)) return false;
    const int m0 = (int)ceil(fmax(lo - tol, 0.0)), m1 = (int)floor(fmin(hi + tol, lim));
    bool found = false;
    for (int m = m0 + coop.lane; m <= m1 && !found; m += coop.n) {
        // signed distance of (x, y): ((y - pa.y) dx - (x - pa.x) dy) / len in [a, c]
        double qlo, qhi;
        if (major_x) {
            const double base = pa.y + ((double)m - pa.x) * dy / dx, k = len / dx;   // y = base + dist * len / dx
            qlo = base + fmin(a * k, c * k);
            qhi = base + fmax(a * k, c * k);
        } else {
            const double base = pa.x + ((double)m - pa.y) * dx / dy, k = -len / dy;  // x = base - dist * len / dy
            qlo = base + fmin(a * k, c * k);
            qhi = base + fmax(a * k, c * k);
        }
        const double other = (double)((major_x ? H : W) - 1);
        const double l = ceil(fmax(qlo - tol, 0.0)), h = floor(fmin(qhi + tol, other));
        found = l <= h;
    }
#if defined(__CUDA_ARCH__)
    if (coop.n > 1) found = __any_sync(0xffffffffu, found);
#endif
    return found;
}

// Triangulates the part [i0, j0] (positions along the arc; arc(t) = site at position t) of a pocket; tri(ia, ib, ic,
// pa, pb, pc) receives the triangles that can hold a pixel (positively oriented). Parts are independent of each other:
// share(i, j) may take the longer child of a split away (another warp works on it) by returning true.
// Returns false when the splitting stack overflowed (cannot happen for arcs below 2^POCKET_STACK vertices).
constexpr int POCKET_STACK = 40;
struct NoShare {
    OFK_HD bool operator()(int, int) const { return false; }
};
// The boundary of the mesh towards the outside as a cyclic chain of sites, the mesh on the left of chain[t] ->
// chain[t + 1]: the frame border in the order above when no point is removed (v == nullptr), else the traced loop
// (trace_outer_loop below).
struct Chain {
    const uint32_t* v;
    int n, H, W;
};
OFK_HD Chain perimeter_chain(int H, int W) { return Chain{nullptr, perim_count(H, W), H, W}; }
OFK_HD uint32_t chain_site(const Chain& c, int t) { return c.v != nullptr ? c.v[t] : perim_site(c.H, c.W, t); }

struct ChainArc {   // position t along the arc that starts at chain index k0 -> site
    Chain c;
    int k0;
    OFK_HD uint32_t operator()(int t) const { return chain_site(c, (k0 + t) % c.n); }
    OFK_HD P2 position(const SiteGrid& g, int t) const { return site_pos(g, (*this)(t)); }
};
// The same arc with the sites and displaced positions of its first `ncached` vertices held in a table (shared memory
// in the pockets kernel): a split scans its part of the arc vertex by vertex, and chain index -> site -> flow load ->
// float64 position is most of what a scan step costs. Same values, fetched instead of recomputed.
struct ChainArcCached {
    Chain c;
    int k0;
    const uint32_t* ids;
    const P2* pos;
    int ncached;
    OFK_HD uint32_t operator()(int t) const { return t < ncached ? ids[t] : chain_site(c, (k0 + t) % c.n); }
    OFK_HD P2 position(const SiteGrid& g, int t) const { return t < ncached ? pos[t] : site_pos(g, (*this)(t)); }
};
template <class ArcFn, class TriFn, class ShareFn>
OFK_HD bool pocket_triangulate(const SiteGrid& g, const ArcFn& arc, int i0, int j0, const Coop& coop, TriFn& tri,
                               ShareFn& share) {
    if (j0 - i0 < 2) return true;
    int lo[POCKET_STACK], hi[POCKET_STACK], sp = 0;
    lo[sp] = i0;
    hi[sp++] = j0;
    while (sp > 0) {
        --sp;
        int i = lo[sp], j = hi[sp];
        while (j - i >= 2) {
            const uint32_t ia = arc(i), ib = arc(j);
            const P2 pa = arc.position(g, i), pb = arc.position(g, j);
            const double ex = dsub(pb.x, pa.x), ey = dsub(pb.y, pa.y);
            ArcBest b;
            b.id = NO_SITE;
            b.t = 0;
            b.p = pa;
            b.omin = b.omax = 0.0;
            b.umin = 0.0;
            b.umax = dfma(ex, ex, dmul(ey, ey));
            for (int t = i + 1 + coop.lane; t < j; t += coop.n) {
                const uint32_t id = arc(t);
                const P2 p = arc.position(g, t);
                const double o = orient(pa, pb, p);
                const double u = dfma(dsub(p.x, pa.x), ex, dmul(dsub(p.y, pa.y), ey));
                b.omin = fmin(b.omin, o);
                b.omax = fmax(b.omax, o);
                b.umin = fmin(b.umin, u);
                b.umax = fmax(b.umax, u);
                if (!(o > 0)) continue;
                if (b.id == NO_SITE || incircle_sign(pa, pb, b.p, p, ia, ib, b.id, id) > 0) {
                    b.id = id;
                    b.t = t;
                    b.p = p;
                }
            }
            arc_reduce(b, pa, pb, ia, ib, coop);
            if (b.id == NO_SITE) break;   // nothing left of the base edge: collinear border
            if (!pocket_may_hold_pixel(pa, pb, b, g.W, g.H, coop)) break;
            tri(ia, ib, b.id, pa, pb, b.p);
            // continue with the shorter part; the longer one goes to another warp or is kept for later (the stack stays
            // logarithmic)
            const int t = b.t;
            const bool left_longer = t - i > j - t;
            const int li = left_longer ? i : t, lj = left_longer ? t : j;
            if (lj - li >= 2 && !share(li, lj)) {
                if (sp >= POCKET_STACK) return false;
                lo[sp] = li;
                hi[sp++] = lj;
            }
            if (left_longer) i = t;
            else j = t;
        }
    }
    return true;
}

// ---------------------------------------------------------------------------------------------- small holes
// Removed points (`consider_mask`) leave faces that no intact cell covers. A face that is a simple polygon of a few
// boundary sites strictly inside the frame, with no site inside -- a single removed point leaves an octagon -- is
// triangulated like a pocket, by one thread: its Delaunay triangles only have its own boundary sites as vertices. The
// thread of the FIRST removed point of a face (smallest index) walks the boundary: from the directed edge a -> b (b the
// neighbour of a in direction k, the face on its left, an intact cell on its right) the boundary continues from b
// along the first direction, turning back from k + 1, that has an intact cell on its right. Faces that are larger,
// touch the frame border, are pinched at a vertex, hold a site or surround an island of intact cells are left to the
// per-pixel search.
#ifndef OFK_HOLE_MAXV
#define OFK_HOLE_MAXV 48
#endif
constexpr int HOLE_MAXV = OFK_HOLE_MAXV;

// cell (ci, cj) = the pixels (ci, cj), (ci, cj+1), (ci+1, cj), (ci+1, cj+1); intact when all four are present
OFK_HD bool cell_intact(const uint8_t* point_mask, int H, int W, int ci, int cj) {
    if (ci < 0 || cj < 0 || ci + 1 >= H || cj + 1 >= W) return false;
    if (point_mask == nullptr) return true;
    const uint8_t* m = point_mask + (size_t)ci * W + cj;
    return m[0] && m[1] && m[W] && m[W + 1];
}

struct HoleLoop {
    int n;
    uint32_t v[HOLE_MAXV];   // boundary sites, the face on the RIGHT of v[t] -> v[t + 1] (the order of a pocket's arc)
    OFK_HD uint32_t operator()(int t) const { return v[t]; }
    OFK_HD P2 position(const SiteGrid& g, int t) const { return site_pos(g, v[t]); }
};

// quadrant q (0..3 = SE, SW, NW, NE) of site (r, c) as a cell
OFK_HD void quadrant_cell(int r, int c, int q, int& ci, int& cj) {
    ci = r - (q >> 1);
    cj = c - (((q + 1) >> 1) & 1);
}

OFK_HD bool hole_loop(const uint8_t* pm, int H, int W, int r, int c, HoleLoop& L) {
    const uint32_t self = (uint32_t)(r * W + c);
    // for the first removed point of a face the two rows above it hold no removed point of the face: the edge
    // (r-1, c-1) -> (r-1, c) has an intact cell above and the face below
    if (r < 2 || c < 1 || !cell_intact(pm, H, W, r - 2, c - 1)) return false;
    const int dr[4] = {0, 1, 0, -1}, dc[4] = {1, 0, -1, 0};
    int ar = r - 1, ac = c - 1, k = 0, n = 0;
    uint32_t fwd_order[HOLE_MAXV];
    int rmin = ar, rmax = ar, cmin = ac, cmax = ac;
    for (;;) {
        if (n >= HOLE_MAXV) return false;
        fwd_order[n++] = (uint32_t)(ar * W + ac);
        rmin = ar < rmin ? ar : rmin; rmax = ar > rmax ? ar : rmax;
        cmin = ac < cmin ? ac : cmin; cmax = ac > cmax ? ac : cmax;
        // the face cell on the left of this edge: inside the frame, and no removed corner before `self`
        int ci, cj;
        quadrant_cell(ar, ac, k, ci, cj);
        if (ci < 0 || cj < 0 || ci + 1 >= H || cj + 1 >= W) return false;
        for (int t = 0; t < 4; ++t) {
            const uint32_t id = (uint32_t)((ci + (t >> 1)) * W + cj + (t & 1));
            if (!pm[id] && id < self) return false;
        }
        const int br = ar + dr[k], bc = ac + dc[k];
        int j = k + 1, turns = 0;
        for (;; --j, ++turns) {
            if (turns > 3) return false;
            quadrant_cell(br, bc, (j + 3) & 3, ci, cj);
            if (cell_intact(pm, H, W, ci, cj)) break;
        }
        ar = br;
        ac = bc;
        k = j & 3;
        if (ar == r - 1 && ac == c - 1 && k == 0) break;
    }
    if (n < 3) return false;
    for (int i = 0; i < n; ++i)       // pinched at a vertex: not a simple polygon
        for (int j = i + 1; j < n; ++j)
            if (fwd_order[i] == fwd_order[j]) return false;
    // an intact cell inside the polygon: the face is a ring around an island of the mesh (four removed points in a
    // pinwheel do that), not a simple polygon. Crossing number of the cell centre against the vertical boundary edges.
    for (int ci = rmin; ci < rmax; ++ci)
        for (int cj = cmin; cj < cmax; ++cj) {
            if (!cell_intact(pm, H, W, ci, cj)) continue;
            int crossings = 0;
            for (int i = 0; i < n; ++i) {
                const uint32_t u = fwd_order[i], v = fwd_order[i + 1 == n ? 0 : i + 1];
                const int ur = (int)(u / (uint32_t)W), uc = (int)(u % (uint32_t)W), vr = (int)(v / (uint32_t)W);
                if (ur != vr && uc > cj && (ur < vr ? ur : vr) == ci) ++crossings;
            }
            if (crossings & 1) return false;
        }
    for (int y = rmin + 1; y < rmax; ++y)   // a site that no intact cell touches may lie inside the face
        for (int x = cmin + 1; x < cmax; ++x)
            if (pm[(size_t)y * W + x] && !cell_intact(pm, H, W, y, x) && !cell_intact(pm, H, W, y, x - 1) &&
                !cell_intact(pm, H, W, y - 1, x - 1) && !cell_intact(pm, H, W, y - 1, x))
                return false;
    L.n = n;
    for (int i = 0; i < n; ++i) L.v[i] = fwd_order[n - 1 - i];
    return true;
}

// triangles of the face whose first removed point is (r, c), if it qualifies
template <class TriFn>
OFK_HD bool hole_fill(const SiteGrid& g, const uint8_t* pm, int r, int c, TriFn& tri) {
    HoleLoop L;
    if (!hole_loop(pm, g.H, g.W, r, c, L)) return false;
    const Coop solo{0, 1};
    NoShare noshare;
    pocket_triangulate(g, L, 0, L.n - 1, solo, tri, noshare);
    return true;
}

// ------------------------------------------------------------------------------------------- triangle rasteriser
// Pixels owned by the positively oriented triangle (p0, p1, p2) with site indices (i0, i1, i2), by the fill rule of
// forward_geom.cuh: an edge evaluated from its smaller-index endpoint, F == 0 given to the triangle that traverses it
// in that direction. Rows are dealt out to the lanes of `coop`; per row the x-interval is bounded conservatively from
// the three edges (long thin pocket triangles have bounding boxes thousands of times their area) and every candidate
// is decided by the exact edge functions. fn(x, y, w0, w1, w2) receives the barycentric weights.
template <class PixelFn>
OFK_HD void raster_triangle(const P2& p0, const P2& p1, const P2& p2, uint32_t i0, uint32_t i1, uint32_t i2, int W,
                            int H, const Coop& coop, PixelFn& fn) {
    const double area2 = orient(p0, p1, p2);
    if (!(area2 > 0.0)) return;
    const double ylo = fmin(p0.y, fmin(p1.y, p2.y)), yhi = fmax(p0.y, fmax(p1.y, p2.y));
    const double xlo = fmin(p0.x, fmin(p1.x, p2.x)), xhi = fmax(p0.x, fmax(p1.x, p2.x));
    if (!(xhi >= 0.0 && yhi >= 0.0 && xlo <= (double)(W - 1) && ylo <= (double)(H - 1))) return;
    const int y0 = (int)ceil(fmax(ylo, 0.0)), y1 = (int)floor(fmin(yhi, (double)(H - 1)));
    const double bx0 = fmax(xlo, 0.0), bx1 = fmin(xhi, (double)(W - 1));
    // edge k is opposite vertex k: (p1 -> p2), (p2 -> p0), (p0 -> p1); canonical endpoints and traversal direction
    const P2* eu[3] = {&p1, &p2, &p0};
    const P2* ev[3] = {&p2, &p0, &p1};
    const bool fwd_dir[3] = {i1 < i2, i2 < i0, i0 < i1};
    const double r = drcp(area2);
    for (int y = y0 + coop.lane; y <= y1; y += coop.n) {
        const double qy = (double)y;
        double xl = bx0, xr = bx1;
        for (int k = 0; k < 3; ++k) {   // inside: dx * (qy - u.y) - dy * (qx - u.x) >= 0
            const double dx = ev[k]->x - eu[k]->x, dy = ev[k]->y - eu[k]->y;
            if (dy == 0.0) continue;
            const double xc = eu[k]->x + dx * (qy - eu[k]->y) / dy;
            const double slack = 1e-6 + 1e-12 * fabs(xc);
            if (dy > 0.0) xr = fmin(xr, xc + slack);
            else xl = fmax(xl, xc - slack);
        }
        if (!(xl <= xr)) continue;
        const int xa = (int)ceil(xl), xb = (int)floor(xr);
        for (int x = xa; x <= xb; ++x) {
            const double qx = (double)x;
            double e[3];
            bool in = true;
            for (int k = 0; k < 3; ++k) {
                if (fwd_dir[k]) {
                    e[k] = edge_canon(*eu[k], *ev[k], qx, qy);
                    in = in && e[k] >= 0.0;
                } else {
                    e[k] = -edge_canon(*ev[k], *eu[k], qx, qy);
                    in = in && e[k] > 0.0;
                }
            }
            if (!in) continue;
            const double w0 = dmul(e[0], r), w1 = dmul(e[1], r);
            fn(x, y, w0, w1, dsub(dsub(1.0, w0), w1));
        }
    }
}

// Pixels exactly on the segment (pa, pb) -- edge function exactly 0, evaluated from the end point with the smaller
// index like everywhere else, end points included: fn(x, y, wa, wb). On a hull edge the fill rule can leave them to
// nobody (the one triangle there may traverse the edge from the larger index to the smaller); they are inside the hull.
template <class LineFn>
OFK_HD void raster_segment(const P2& pa, const P2& pb, int W, int H, const Coop& coop, LineFn& fn) {
    const double xlo = fmin(pa.x, pb.x), xhi = fmax(pa.x, pb.x), ylo = fmin(pa.y, pb.y), yhi = fmax(pa.y, pb.y);
    if (!(xhi >= 0.0 && yhi >= 0.0 && xlo <= (double)(W - 1) && ylo <= (double)(H - 1))) return;
    const int x0 = (int)ceil(fmax(xlo, 0.0)), x1 = (int)floor(fmin(xhi, (double)(W - 1)));
    const int y0 = (int)ceil(fmax(ylo, 0.0)), y1 = (int)floor(fmin(yhi, (double)(H - 1)));
    const double dx = dsub(pb.x, pa.x), dy = dsub(pb.y, pa.y);
    const double len2 = dfma(dx, dx, dmul(dy, dy));
    if (!(len2 > 0.0)) return;
    const bool steep = fabs(dy) > fabs(dx);
    // one candidate per row (steep) or per column: the lattice point next to the line
    const int n = steep ? y1 - y0 + 1 : x1 - x0 + 1;
    for (int t = coop.lane; t < n; t += coop.n) {
        int x, y;
        if (steep) {
            y = y0 + t;
            x = (int)rint(pa.x + dx * ((double)y - pa.y) / dy);
        } else {
            x = x0 + t;
            y = (int)rint(pa.y + dy * ((double)x - pa.x) / dx);
        }
        if (x < x0 || x > x1 || y < y0 || y > y1) continue;
        if (edge_canon(pa, pb, (double)x, (double)y) != 0.0) continue;
        const double rx = dsub((double)x, pa.x), ry = dsub((double)y, pa.y);
        double wb = dfma(rx, dx, dmul(ry, dy)) / len2;
        wb = wb < 0.0 ? 0.0 : (wb > 1.0 ? 1.0 : wb);
        fn(x, y, dsub(1.0, wb), wb);
    }
}

// The pixels exactly on border edges t0 <= t < t1 (edge t joins border sites t and t + 1) that no intact cell
// produced: seg(ia, ib, pa, pb, coop) gets the end points ordered by index. They come before the triangles of the
// pockets (which leave produced pixels alone), the hull edge of a pocket -- pocket_chord -- after them.
template <class SegFn>
OFK_HD void pocket_border_edges(const SiteGrid& g, const Chain& ch, int t0, int t1, int stride, SegFn& seg) {
    const Coop solo{0, 1};
    for (int t = t0; t < t1; t += stride) {
        const uint32_t ia = chain_site(ch, t), ib = chain_site(ch, t + 1 == ch.n ? 0 : t + 1);
        const P2 pa = site_pos(g, ia), pb = site_pos(g, ib);
        if (ia < ib) seg(ia, ib, pa, pb, solo);
        else seg(ib, ia, pb, pa, solo);
    }
}

template <class SegFn>
OFK_HD void pocket_chord(const SiteGrid& g, const Chain& ch, int k0, int k1, const Coop& coop, SegFn& seg) {
    if (((k1 - k0) % ch.n + ch.n) % ch.n < 2) return;
    const uint32_t ia = chain_site(ch, k0), ib = chain_site(ch, k1);
    const P2 pa = site_pos(g, ia), pb = site_pos(g, ib);
    if (ia < ib) seg(ia, ib, pa, pb, coop);
    else seg(ib, ia, pb, pa, coop);
}

// ---------------------------------------------------------------------------------------- outer boundary of a mask
// With removed points the mesh ends where the point mask does. A forward pass leaves exactly such masks behind (valid
// inside the hull of the resampled points: a rotated frame with staircase edges), and the next pass of a chain
// (switch_ref, modes 1 / 2) takes them as its point mask: between the staircase and its hull lie hundreds of small
// pockets per frame. The boundary is walked like the boundary of a hole (hole_loop), from the first valid site in
// raster order, whose upper side faces the outside; the result is stored reversed, mesh on the left, like the
// frame border. Gives up (returns -1: per-pixel search) when the chain does not fit, the start is a site without a
// cell, or the mesh is pinched at a visited vertex (two separate open sectors: the chain would not be a simple
// polygon). Sites without any cell inside the outside face make the pockets more than polygons: the caller checks
// for them separately (any_isolated_site).
OFK_HD int trace_outer_loop(const uint8_t* pm, int H, int W, uint32_t first_valid, uint32_t* out, int cap) {
    if (pm == nullptr || H < 2 || W < 2 || first_valid >= (uint32_t)H * (uint32_t)W) return -1;
    const int r0 = (int)(first_valid / (uint32_t)W), c0 = (int)(first_valid % (uint32_t)W);
    const int dr[4] = {0, 1, 0, -1}, dc[4] = {1, 0, -1, 0};
    auto quad_intact = [&](int r, int c, int q) {
        int ci, cj;
        quadrant_cell(r, c, q & 3, ci, cj);
        return cell_intact(pm, H, W, ci, cj);
    };
    // the open sector that holds the quadrants above the start site begins after an intact quadrant
    int k0 = 2, turns = 0;
    while (!quad_intact(r0, c0, k0 + 3)) {
        --k0;
        if (++turns > 3) return -1;   // no cell touches the first site
    }
    k0 &= 3;
    int ar = r0, ac = c0, k = k0, n = 0;
    for (;;) {
        if (n >= cap) return -1;
        const bool q0 = quad_intact(ar, ac, 0), q1 = quad_intact(ar, ac, 1), q2 = quad_intact(ar, ac, 2),
                   q3 = quad_intact(ar, ac, 3);
        if ((q0 && q2 && !q1 && !q3) || (q1 && q3 && !q0 && !q2)) return -1;   // pinched
        out[n++] = (uint32_t)(ar * W + ac);
        const int br = ar + dr[k], bc = ac + dc[k];
        int j = k + 1;
        turns = 0;
        while (!quad_intact(br, bc, j + 3)) {
            --j;
            if (++turns > 3) return -1;
        }
        ar = br;
        ac = bc;
        k = j & 3;
        if (ar == r0 && ac == c0 && k == k0) break;
    }
    if (n < 3) return -1;
    for (int i = 0, j = n - 1; i < j; ++i, --j) {   // the walk has the outside on its left: reversed
        const uint32_t t = out[i];
        out[i] = out[j];
        out[j] = t;
    }
    return n;
}

// a valid site that no intact cell touches (all four quadrants open)
OFK_HD bool site_is_isolated(const uint8_t* pm, int H, int W, int r, int c) {
    return !cell_intact(pm, H, W, r, c) && !cell_intact(pm, H, W, r, c - 1) && !cell_intact(pm, H, W, r - 1, c - 1) &&
           !cell_intact(pm, H, W, r - 1, c);
}

// a valid site is a boundary site when it sits on the frame border or one of its 8 neighbours has been removed
OFK_HD bool is_boundary_site(const uint8_t* point_mask, int H, int W, int row, int col) {
    if (point_mask != nullptr && !point_mask[(size_t)row * W + col]) return false;
    if (row == 0 || col == 0 || row == H - 1 || col == W - 1) return true;
    if (point_mask == nullptr) return false;
    const uint8_t* m = point_mask + (size_t)row * W + col;
    return !(m[-W - 1] && m[-W] && m[-W + 1] && m[-1] && m[1] && m[W - 1] && m[W] && m[W + 1]);
}

}  // namespace fwd
}  // namespace ofk
