// TEST INFRASTRUCTURE -- host build of the forward-resampling algorithm of oflibnumpy_b200/csrc/forward_geom.cuh and
// forward_irregular.cuh (the very same header code the CUDA kernels in forward_s.cu execute), run serially on the CPU
// so that the CPU test-suite can check the ALGORITHM against outputs of the unmodified reference (tests/golden) without
// a GPU. It is compiled by tests/test_forward_hostsim.py into a scratch directory; the package never loads it and no
// product path can reach it (the product path fails loudly without the CUDA library).
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../oflibnumpy_b200/csrc/forward_irregular.cuh"

using namespace ofk::fwd;

namespace {

struct Frame {
    const float* payload;
    int C;
    const float* flow;
    float sign;
    const uint8_t* payload_mask;
    const uint8_t* point_mask;
    float* out;
    uint8_t* out_mask;
    int rule_strict;
    int H, W;
    uint8_t* cover;
};

struct EmitHost {
    const Frame& f;
    int i, j;   // cell
    long long count;
    void operator()(int x, int y, int k0, int k1, int k2, double w0, double w1, double w2) {
        const int W = f.W;
        const size_t v0 = (size_t)(i + (k0 >> 1)) * W + j + (k0 & 1), v1 = (size_t)(i + (k1 >> 1)) * W + j + (k1 & 1),
                     v2 = (size_t)(i + (k2 >> 1)) * W + j + (k2 & 1);
        const size_t px = (size_t)y * W + x;
        const uint8_t* pm = f.payload_mask;
        interp_store(f.payload + v0 * f.C, f.payload + v1 * f.C, f.payload + v2 * f.C, pm ? pm[v0] != 0 : true,
                     pm ? pm[v1] != 0 : true, pm ? pm[v2] != 0 : true, w0, w1, w2, f.C, f.out + px * f.C,
                     f.out_mask ? f.out_mask + px : nullptr, f.rule_strict);
        f.cover[px] += 1;   // counts how many triangles produced the pixel: the fill rule promises exactly one
        ++count;
    }
};

}  // namespace

// stats: [0] pixels from intact cells, [1] irregular pixels located, [2] outside the hull (located), [3] walk failures,
//        [4] rejected by the hull pre-filter, [5] folded cells, [6] pixels produced more than once, [7] boundary sites,
//        [10] 1 when the frame folds and was triangulated as a whole
// A frame with a folded cell (a displaced cell that is not a positively oriented quadrilateral) is not a mesh of its
// cells: every kept point becomes a site and every pixel is located in their Delaunay triangulation, as on the device.
extern "C" int fwd_hostsim(const float* payload, int C, const float* flow, float sign, const uint8_t* payload_mask,
                           const uint8_t* point_mask, float* out, uint8_t* out_mask, int rule_strict, int H, int W,
                           int use_prefilter, double flip_tol, long long* stats) {
    const int use_hints = (use_prefilter & 2) != 0;
    const int flags = use_prefilter;
    use_prefilter &= 1;
    std::vector<uint8_t> cover((size_t)H * W, 0);
    Frame f{payload, C, flow, sign, payload_mask, point_mask, out, out_mask, rule_strict, H, W, cover.data()};
    memset(stats, 0, 12 * sizeof(long long));
    // ---- regular part: intact cells
    for (int i = 0; i + 1 < H; ++i) {
        for (int j = 0; j + 1 < W; ++j) {
            const size_t o = (size_t)i * W + j;
            if (point_mask && !(point_mask[o] && point_mask[o + 1] && point_mask[o + W] && point_mask[o + W + 1]))
                continue;
            const P2 a = displaced(flow[2 * o], flow[2 * o + 1], i, j, sign);
            const P2 b = displaced(flow[2 * (o + 1)], flow[2 * (o + 1) + 1], i, j + 1, sign);
            const P2 c = displaced(flow[2 * (o + W)], flow[2 * (o + W) + 1], i + 1, j, sign);
            const P2 d = displaced(flow[2 * (o + W + 1)], flow[2 * (o + W + 1) + 1], i + 1, j + 1, sign);
            double area2[2];
            const int diag = cell_diagonal(a, b, c, d, area2, flip_tol);
            if (diag < 0) {
                ++stats[5];
                continue;
            }
            EmitHost e{f, i, j, 0};
            raster_cell(a, b, c, d, diag, area2, W, H, e);
            stats[0] += e.count;
        }
    }
    for (size_t k = 0; k < cover.size(); ++k)
        if (cover[k] > 1) ++stats[6];
    const bool whole = stats[5] > 0;
    if (whole) {
        stats[10] = 1;
        stats[0] = stats[6] = 0;
        std::fill(cover.begin(), cover.end(), 0);
    }
    // ---- boundary sites, binned by position
    SiteGrid g;
    g.H = H;
    g.W = W;
    g.nbx = grid_bins(W);
    g.nby = grid_bins(H);
    g.ncx = grid_coarse(g.nbx);
    g.ncy = grid_coarse(g.nby);
    g.flow = flow;
    g.sign = sign;
    g.inv_w = grid_inv(W);
    const int nb = grid_slots(g.nbx, g.nby);
    std::vector<uint32_t> start(nb + 1, 0), sites;
    std::vector<unsigned long long> occ((size_t)g.ncx * g.ncy, 0);
    std::vector<uint32_t> ids;
    for (int i = 0; i < H; ++i)
        for (int j = 0; j < W; ++j)
            if (whole ? (point_mask == nullptr || point_mask[(size_t)i * W + j] != 0)
                      : is_boundary_site(point_mask, H, W, i, j))
                ids.push_back((uint32_t)(i * W + j));
    stats[7] = (long long)ids.size();
    std::vector<int> bin_of(ids.size());
    for (size_t k = 0; k < ids.size(); ++k) {
        const uint32_t id = ids[k];
        const P2 p = displaced(flow[2 * (size_t)id], flow[2 * (size_t)id + 1], (int)(id / W), (int)(id % W), sign);
        const int bx = bin_coord(p.x, g.nbx), by = bin_coord(p.y, g.nby);
        bin_of[k] = bin_index(g.nbx, bx, by);
        ++start[bin_of[k] + 1];
        occ[(by >> COARSE_SHIFT) * g.ncx + (bx >> COARSE_SHIFT)] |=
            1ull << (((by & ((1 << COARSE_SHIFT) - 1)) << COARSE_SHIFT) | (bx & ((1 << COARSE_SHIFT) - 1)));
    }
    for (int b = 0; b < nb; ++b) start[b + 1] += start[b];
    sites.resize(ids.size());
    {
        std::vector<uint32_t> cur(start.begin(), start.end() - 1);
        // filled back to front: the device fills with atomics in arbitrary order, the result must not depend on it
        for (size_t k = ids.size(); k-- > 0;) sites[cur[bin_of[k]]++] = ids[k];
    }
    g.bin_start = start.data();
    g.occ = occ.data();
    g.sites = sites.data();
    // ---- hull pre-filter
    HullInfo hull;
    HullDirs dirs;
    for (int k = 0; k < HULL_DIRS; ++k) {
        dirs.dx[k] = cos(2.0 * M_PI * k / HULL_DIRS);
        dirs.dy[k] = sin(2.0 * M_PI * k / HULL_DIRS);
    }
    hull_build_serial(g, (uint32_t)ids.size(), dirs, hull);
    std::vector<P2> opos;
    std::vector<uint32_t> oids;
    for (size_t k = 0; k < ids.size(); ++k) {
        const P2 p = site_pos(g, ids[k]);
        if (hull_outer_candidate(hull, p)) {
            opos.push_back(p);
            oids.push_back(ids[k]);
        }
    }
    static HullPoly poly;
    hull_wrap_serial(opos.data(), oids.data(), (int)opos.size(), poly);
    if (!use_prefilter) {
        hull.m = 0;
        poly.ok = 0;
    }
    // ---- hull pockets: between the boundary chain of the mesh (the frame border, or the traced outer boundary of the
    // point mask) and its hull, triangulated arc by arc, rasterised directly
    std::vector<uint32_t> chain_store;
    std::vector<int> hull_pos;
    Chain ch{nullptr, 0, H, W};
    bool have_chain = false;
    if (!whole && poly.ok && H >= 3 && W >= 3 && (flags & 4) == 0) {
        bool removed_any = false;
        if (point_mask != nullptr)
            for (size_t k = 0; k < (size_t)H * W && !removed_any; ++k) removed_any = point_mask[k] == 0;
        if (!removed_any) {
            ch = perimeter_chain(H, W);
            hull_pos.resize(poly.m);
            have_chain = true;
            for (int e = 0; e < poly.m; ++e) {
                hull_pos[e] = perim_index(H, W, poly.id[e]);
                if (hull_pos[e] < 0) have_chain = false;
            }
        } else if ((flags & 16) == 0) {
            uint32_t first = 0xffffffffu;
            bool isolated = false;
            for (int r = 0; r < H; ++r)
                for (int c = 0; c < W; ++c)
                    if (point_mask[(size_t)r * W + c]) {
                        if (first == 0xffffffffu) first = (uint32_t)(r * W + c);
                        isolated = isolated || site_is_isolated(point_mask, H, W, r, c);
                    }
            chain_store.resize(4 * (size_t)(H + W));
            const int n = isolated ? -1 : trace_outer_loop(point_mask, H, W, first, chain_store.data(), (int)chain_store.size());
            if (n > 0) {
                ch = Chain{chain_store.data(), n, H, W};
                hull_pos.assign(poly.m, -1);
                for (int t = 0; t < n; ++t)
                    for (int e = 0; e < poly.m; ++e)
                        if (poly.id[e] == chain_store[t] && hull_pos[e] < 0) hull_pos[e] = t;
                have_chain = true;
                for (int e = 0; e < poly.m; ++e)
                    if (hull_pos[e] < 0) have_chain = false;
            }
        }
    }
    if (have_chain) {
        ++stats[9];
        const Coop solo{0, 1};
        const uint8_t* pm = payload_mask;
        auto seg = [&](uint32_t ia, uint32_t ib, const P2& pa, const P2& pb, const Coop& co) {
            auto pixel = [&](int x, int y, double wa, double wb) {
                const size_t px = (size_t)y * W + x;
                if (cover[px]) return;
                cover[px] = 3;
                ++stats[1];
                interp_store(payload + (size_t)ia * C, payload + (size_t)ib * C, payload + (size_t)ib * C,
                             pm ? pm[ia] != 0 : true, pm ? pm[ib] != 0 : true, pm ? pm[ib] != 0 : true, wa, wb, 0.0, C,
                             out + px * C, out_mask ? out_mask + px : nullptr, rule_strict);
            };
            raster_segment(pa, pb, W, H, co, pixel);
        };
        pocket_border_edges(g, ch, 0, ch.n, 1, seg);
        for (int e = 0; e < poly.m; ++e) {
            const int k0 = hull_pos[e], k1 = hull_pos[e + 1 == poly.m ? 0 : e + 1];
            auto tri = [&](uint32_t ia, uint32_t ib, uint32_t ic, const P2& pa, const P2& pb, const P2& pc) {
                auto pixel = [&](int x, int y, double w0, double w1, double w2) {
                    const size_t px = (size_t)y * W + x;
                    // a pixel within rounding of the displaced border can be claimed from both sides (the sliver's
                    // edges are chords, not the border edge the cell was tested against): the cell keeps it
                    if (cover[px]) {
                        if (cover[px] == 2) ++stats[6];
                        return;
                    }
                    cover[px] = 2;
                    ++stats[1];
                    interp_store(payload + (size_t)ia * C, payload + (size_t)ib * C, payload + (size_t)ic * C,
                                 pm ? pm[ia] != 0 : true, pm ? pm[ib] != 0 : true, pm ? pm[ic] != 0 : true, w0, w1, w2, C,
                                 out + px * C, out_mask ? out_mask + px : nullptr, rule_strict);
                };
                raster_triangle(pa, pb, pc, ia, ib, ic, W, H, solo, pixel);
            };
            NoShare noshare;
            const ChainArc arc{ch, k0};
            if (!pocket_triangulate(g, arc, 0, ((k1 - k0) % ch.n + ch.n) % ch.n, solo, tri, noshare)) ++stats[3];
            pocket_chord(g, ch, k0, k1, solo, seg);
        }
    }
    // ---- small faces left by removed points: triangulated by the thread of their first removed point
    if (!whole && point_mask != nullptr && (flags & 8) == 0) {
        const uint8_t* pm = payload_mask;
        for (int r = 0; r < H; ++r)
            for (int c = 0; c < W; ++c) {
                if (point_mask[(size_t)r * W + c]) continue;
                auto tri = [&](uint32_t ia, uint32_t ib, uint32_t ic, const P2& pa, const P2& pb, const P2& pc) {
                    auto pixel = [&](int x, int y, double w0, double w1, double w2) {
                        const size_t px = (size_t)y * W + x;
                        if (cover[px]) {
                            if (cover[px] == 2) ++stats[6];
                            return;
                        }
                        cover[px] = 2;
                        ++stats[1];
                        interp_store(payload + (size_t)ia * C, payload + (size_t)ib * C, payload + (size_t)ic * C,
                                     pm ? pm[ia] != 0 : true, pm ? pm[ib] != 0 : true, pm ? pm[ic] != 0 : true, w0, w1,
                                     w2, C, out + px * C, out_mask ? out_mask + px : nullptr, rule_strict);
                    };
                    raster_triangle(pa, pb, pc, ia, ib, ic, W, H, Coop{0, 1}, pixel);
                };
                if (hole_fill(g, point_mask, r, c, tri)) ++stats[8];
            }
    }
    // ---- irregular part
    for (int y = 0; y < H; ++y) {
        uint32_t hint[3] = {0, 0, 0};
        int hint_x = -2;
        for (int x = 0; x < W; ++x) {
            const size_t px = (size_t)y * W + x;
            if (cover[px]) continue;
            P2 q;
            q.x = x;
            q.y = y;
            uint32_t vid[3];
            double w[3];
            int st;
            if (hull_rejects(hull, q) || (poly.ok && !inside_hull(poly, q))) {
                st = LOC_OUTSIDE;
                ++stats[4];
            } else {
                st = (use_hints && hint_x == x - 1) ? locate_hinted(g, q, hint, vid, w) : locate(g, q, vid, w);
                if (st == LOC_FOUND) {
                    hint[0] = vid[0]; hint[1] = vid[1]; hint[2] = vid[2];
                    hint_x = x;
                }
                if (st == LOC_OUTSIDE) ++stats[2];
                if (st == LOC_FAILED) ++stats[3];
                if (st == LOC_FOUND) ++stats[1];
            }
            if (st == LOC_FOUND) {
                const uint8_t* pm = payload_mask;
                interp_store(payload + (size_t)vid[0] * C, payload + (size_t)vid[1] * C, payload + (size_t)vid[2] * C,
                             pm ? pm[vid[0]] != 0 : true, pm ? pm[vid[1]] != 0 : true, pm ? pm[vid[2]] != 0 : true,
                             w[0], w[1], w[2], C, out + px * C, out_mask ? out_mask + px : nullptr, rule_strict);
            } else {
                for (int c = 0; c < C; ++c) out[px * C + c] = 0.f;
                if (out_mask) out_mask[px] = 0;
            }
        }
    }
    return 0;
}
