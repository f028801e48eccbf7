// Fused flow composition, mode 3, for sm_100a: warp-specialised, TMA-staged kernel (the default path of ofk_combine3).
//
//   ref 't' : out[p] = B[p] + Q(A, p - B[p]);   out_mask[p] = Bm[p] & strict(Am at the taps)     (P = B, G = A, sign -1)
//   ref 's' : out[p] = A[p] + Q(B, p + A[p]);   out_mask[p] = Am[p] & strict(Bm at the taps)     (P = A, G = B, sign +1)
//
// Q is the cv2.remap float32 bilinear sample (1/32-px coordinates, zero border); reference: flow_class.py:1411-1422.
//
// CTA = 1 producer warp + 8 consumer warps, persistent over 32x32 output tiles, 2 CTAs per SM.
//   producer : TMA-loads the pointwise operand tile (P, Pm) two tiles ahead; when a P tile has landed it estimates the
//              bounding box of the tile's sample positions from the tile perimeter, and TMA-loads that 48x48 box of
//              the gathered operand (G, Gm) into a box stage. The hardware zero fill outside the frame is exactly
//              cv2.remap's BORDER_CONSTANT(0) and "mask invalid outside the frame".
//   consumers: wait for the box, gather the four taps of every pixel from shared memory (32-bit offsets, no bounds
//              tests, no border path), blend with packed f32x2 arithmetic in cv2.remap's rounding sequence, write the
//              result over the P tile in place and hand the warp's four rows to a TMA store (clipped at the frame
//              border by the hardware).
// Pixels whose taps are not covered by the box (estimate too small, discontinuous or noisy flows) fetch their taps from
// global memory instead, with the same arithmetic, so the result never depends on the quality of the estimate. HBM traffic is the algorithmic 27 B/px:
// P and the output stream once; the boxes overlap, but the overlap is served by L2.
//
// The zero tests gating the reference's early exits (flow_class.py:1338-1354) are not part of the hot loop: a probe
// kernel looks at a sparse sample of every operand (almost always enough to prove "not zero"), a scan kernel reads the
// operands completely only for frames the probe could not decide, and combine3_fixup (combine3.cu) applies the exits.
#include <stdlib.h>

#include <type_traits>

#include "combine3_device.cuh"
#include "ws_common.cuh"

namespace ofk {
namespace c3ws {
using namespace ws;


constexpr int TS = 32;
constexpr int BW = 48, BH = 48;   // vector box (pixels)
constexpr int BMW = 64;           // mask box width (bytes): start is aligned down to 16
constexpr int NCW = 8;            // consumer warps

template <int NP, int NB>
struct Smem {
    struct PStage {
        float2 p[TS * TS];
        uint8_t pm[TS * TS];
    };
    struct BStage {
        float2 v[BH * BW];
        uint8_t m[BH * BMW];
    };
    alignas(128) PStage ps[NP];
    alignas(128) BStage bs[NB];
    alignas(16) int4 binfo[NB][2];   // {vx0, vx0 - mx0, by0, -}, {tx0, ty0, n, -}
    uint64_t pfull[NP], pempty[NP], bfull[NB], bempty[NB];
    uint32_t sink[NCW];              // scratch words of mbar_arrive_after, one per consumer warp
};

struct Maps {
    CUtensorMap p, pm, gb, gmb, ov, om;
};

// packed f32x2 arithmetic (sm_100): both halves are IEEE round-to-nearest, no contraction
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float2 unpack2(uint64_t v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// a * b rounded once: fma with a (-0, -0) addend the compiler cannot see through (kernel parameter). A plain
// mul.rn.f32x2 feeding add.rn.f32x2 is contracted into FFMA2 by ptxas 12.9 in spite of the .rn qualifiers, which would
// change the rounding sequence of cv2.remap.
__device__ __forceinline__ uint64_t mul2_nofuse(uint64_t a, uint64_t b, uint64_t negzero2) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(negzero2));
    return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

__device__ __forceinline__ void quant(float X, int& i, int& f) {
    const int bits = __float_as_int(__fmaf_rn(X, 32.0f, 12582912.0f)) - 0x4B400000;
    i = bits >> 5;
    f = bits & 31;
}

// What pixel j of this thread writes (EPI_* of combine3_device.cuh): p = P[p], s = Q(G, ...) packed, v = its validity
// byte. The consistency epilogue writes its byte over the P mask tile (the mask store) and keeps the valid byte in vb.
template <int EPI>
__device__ __forceinline__ void epilogue(float2* prow, uint8_t* mrow, int j, uint64_t p, uint64_t s, unsigned v,
                                         unsigned& vb, const EpiArgs<EPI>& epi) {
    if constexpr (EPI == EPI_CONSIST) {
        const float2 w = unpack2(p), q = unpack2(s);
        mrow[j * TS] = (uint8_t)(v & fb_consistent(w.x, w.y, q.x, q.y, epi.a1, epi.a2));
        vb = v;
    } else {
        *reinterpret_cast<uint64_t*>(prow + j * TS) = EPI == EPI_COMPOSE ? add2(p, s) : s;
        mrow[j * TS] = (uint8_t)v;
    }
}
// The consistency epilogue's valid bytes go out through the vector map slot, staged in the warp's own 4 P vector rows
// (4 x 32 bytes from the start of its first row). Lanes overwrite vectors of other lanes there, so the warp first makes
// sure that every lane has read its vectors. prow: this lane's first pixel in the P stage.
template <int EPI>
__device__ __forceinline__ void stage_valid(float2* prow, const unsigned (&vb)[4], const EpiArgs<EPI>& epi) {
    if constexpr (EPI == EPI_CONSIST) {
        __syncwarp();
        if (epi.valid != nullptr) {
            const unsigned lane = threadIdx.x & 31;
            uint8_t* vrow = reinterpret_cast<uint8_t*>(prow - lane) + lane;
#pragma unroll
            for (int j = 0; j < 4; ++j) vrow[j * TS] = (uint8_t)vb[j];
        }
    }
}

// The global-tap path (out of line, see mixed_rows): taps of a warp's 4 x 32 pixels, all requested before the first
// use -- from the box for the pixels it covers, from global memory for the others, predicated per tap on "inside the
// frame" (zero border, mask invalid outside) -- then validity, release of the box, blend: one memory round trip per
// warp and tile and the same arithmetic as the main path, so the result never depends on the box estimate.
template <bool MASKS, int EPI, class BStage>
__device__ __forceinline__ void sample_rows_mixed(const BStage& bs, float2* prow, uint8_t* mrow, const uint64_t (&p)[4],
                                            const unsigned (&pm)[4], const int (&dx)[4], const int (&dy)[4],
                                            const int (&fa)[4], const int (&fb)[4], int4 info, int n,
                                            const float2* __restrict__ G, const uint8_t* __restrict__ Gm, int H, int W,
                                            uint64_t negzero2, uint64_t* bempty, uint32_t* sink, unsigned lane,
                                            const EpiArgs<EPI>& epi) {
    const uint64_t one2 = pack2(1.0f, 1.0f);
    unsigned vb[4];
    uint64_t t[4][4];
    unsigned m[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const bool inbox = (unsigned)dx[j] < (unsigned)(BW - 1) && (unsigned)dy[j] < (unsigned)(BH - 1);
        if (inbox) {
            const uint64_t* v = reinterpret_cast<const uint64_t*>(bs.v) + (dy[j] * BW + dx[j]);
            t[j][0] = v[0]; t[j][1] = v[1]; t[j][2] = v[BW]; t[j][3] = v[BW + 1];
            if (MASKS) {
                const uint8_t* mm = bs.m + (dy[j] * BMW + dx[j] + info.y);
                m[j][0] = mm[0]; m[j][1] = mm[1]; m[j][2] = mm[BMW]; m[j][3] = mm[BMW + 1];
            }
        } else {
            // integer coordinates from the fast quantiser: exact for |X| < 2^17, far outside the frame otherwise
            const int ix = dx[j] + info.x, iy = dy[j] + info.z;
            const bool x0 = (unsigned)ix < (unsigned)W, x1 = (unsigned)(ix + 1) < (unsigned)W;
            const bool y0 = (unsigned)iy < (unsigned)H, y1 = (unsigned)(iy + 1) < (unsigned)H;
            const long long o = (long long)n * ((long long)H * W) + ((long long)iy * W + ix);
            const uint64_t* g = reinterpret_cast<const uint64_t*>(G) + o;
            t[j][0] = (x0 && y0) ? __ldg(g) : 0ull;
            t[j][1] = (x1 && y0) ? __ldg(g + 1) : 0ull;
            t[j][2] = (x0 && y1) ? __ldg(g + W) : 0ull;
            t[j][3] = (x1 && y1) ? __ldg(g + W + 1) : 0ull;
            if (MASKS) {
                const uint8_t* gm = Gm + o;
                m[j][0] = (x0 && y0) ? __ldg(gm) : 0u;
                m[j][1] = (x1 && y0) ? __ldg(gm + 1) : 0u;
                m[j][2] = (x0 && y1) ? __ldg(gm + W) : 0u;
                m[j][3] = (x1 && y1) ? __ldg(gm + W + 1) : 0u;
            }
        }
    }
    // validity and a reduction over every tap first: once they are known all taps of this warp have left the box and
    // the stage can be handed back to the producer while the blend is still running
    unsigned strict[4], dep = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned a = fa[j], bb = fb[j];
        const unsigned ha = min(a, 1u), hb = min(bb, 1u);      // 1 where the right / lower taps have weight
        if (MASKS) {
            strict[j] = m[j][0] & (m[j][1] | ~ha) & (m[j][2] | ~hb) & (m[j][3] | ~(ha & hb)) & pm[j];
        } else {
            const int ix = dx[j] + info.x, iy = dy[j] + info.z;
            strict[j] = (ix >= 0 && iy >= 0 && (ix + 1 < W || (a == 0 && ix < W)) &&
                         (iy + 1 < H || (bb == 0 && iy < H))) ? 1u : 0u;
        }
        // every tap feeds the release below (bit 8, masked off when the validity byte is stored): the loads may be
        // issued in any order, so "the value loaded last" is not something the source can name
        strict[j] |= (unsigned)((t[j][0] | t[j][1] | t[j][2] | t[j][3]) >> 63) << 8;
        dep |= strict[j];
    }
    dep = __reduce_or_sync(0xffffffffu, dep);
    if (lane == 0) mbar_arrive_after(bempty, dep, sink);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const unsigned a = fa[j], bb = fb[j];
        const float ffa = (float)a * (1.0f / 32.0f), ffb = (float)bb * (1.0f / 32.0f);
        const uint64_t fa2 = pack2(ffa, ffa), fb2 = pack2(ffb, ffb);
        const uint64_t na2 = add2(one2, fa2 ^ 0x8000000080000000ull), nb2 = add2(one2, fb2 ^ 0x8000000080000000ull);
        uint64_t accv = mul2_nofuse(t[j][0], mul2(na2, nb2), negzero2);
        accv = add2(accv, mul2_nofuse(t[j][1], mul2(fa2, nb2), negzero2));
        accv = add2(accv, mul2_nofuse(t[j][2], mul2(na2, fb2), negzero2));
        accv = add2(accv, mul2_nofuse(t[j][3], mul2(fa2, fb2), negzero2));
        epilogue<EPI>(prow, mrow, j, p[j], accv, strict[j] & 1u, vb[j], epi);
    }
    stage_valid<EPI>(prow, vb, epi);
}

// this thread's four pixels of a tile: operand values, sample positions relative to the box, 1/32-px fractions;
// returns whether all of them are covered by the box
template <bool MASKS>
__device__ __forceinline__ bool prepare_rows(const float2* prow, const uint8_t* mrow, float sign, float xg, float yg,
                                             int4 info, uint64_t (&p)[4], unsigned (&pm)[4], int (&dx)[4], int (&dy)[4],
                                             int (&fa)[4], int (&fb)[4]) {
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        p[j] = *reinterpret_cast<const uint64_t*>(prow + j * TS);
        pm[j] = MASKS ? mrow[j * TS] : 1u;
        const float2 pv = unpack2(p[j]);
        const float X = __fmaf_rn(sign, pv.x, xg), Y = __fmaf_rn(sign, pv.y, yg + (float)j);
        int ix, iy;
        quant(X, ix, fa[j]);
        quant(Y, iy, fb[j]);
        dx[j] = ix - info.x;
        dy[j] = iy - info.z;
        // Covered by the box? Everything else is decided per pixel. No range test is needed for the fast quantiser:
        // it is exact for |X| < 2^17, and beyond that (or for NaN / Inf) the integer it produces is far outside
        // [-2^16, 2^16], so such a pixel can never pass the box test (frames are smaller than 32768).
        ok = ok && (unsigned)dx[j] < (unsigned)(BW - 1) && (unsigned)dy[j] < (unsigned)(BH - 1);
    }
    return ok;
}

// The rare path, out of line so that it does not weigh on the register allocation of the kernel's main loop: redoes the
// preparation from shared memory and samples with sample_rows_mixed.
static __device__ unsigned long long g_mixed_warp_tiles;   // test hook: how often the out-of-line path ran (per warp and tile)

// (epi: the EpiArgs of the consistency epilogue, nothing otherwise, so that the other kernels keep their calls)
template <int EPI>
__device__ __forceinline__ EpiArgs<EPI> epi_args() { return EpiArgs<EPI>{}; }
template <int EPI>
__device__ __forceinline__ EpiArgs<EPI> epi_args(const EpiArgs<EPI>& e) { return e; }

template <bool MASKS, int EPI, class SM, class... E>
__device__ __noinline__ void mixed_rows(typename SM::PStage* ps, const typename SM::BStage* bs, uint64_t* bempty,
                                        uint32_t* sink, int4 info, int4 tile, const float2* __restrict__ G,
                                        const uint8_t* __restrict__ Gm, float sign, int H, int W, uint64_t negzero2,
                                        E... epi) {
    const unsigned lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    if (lane == 0) atomicAdd(&g_mixed_warp_tiles, 1ull);
    float2* prow = ps->p + ((int)wrp * 4 * TS + lane);
    uint8_t* mrow = ps->pm + ((int)wrp * 4 * TS + lane);
    uint64_t p[4];
    unsigned pm[4];
    int dx[4], dy[4], fa[4], fb[4];
    prepare_rows<MASKS>(prow, mrow, sign, (float)(tile.x + (int)lane), (float)(tile.y + (int)wrp * 4), info, p, pm, dx, dy,
                        fa, fb);
    sample_rows_mixed<MASKS, EPI>(*bs, prow, mrow, p, pm, dx, dy, fa, fb, info, tile.z, G, Gm, H, W, negzero2, bempty,
                                  sink, lane, epi_args<EPI>(epi...));
}

// EPI (combine3_device.cuh): EPI_COMPOSE out = P + Q(G, ...) (composition); EPI_SAMPLE out = Q(G, ...) alone (Flow.apply
// of a flow: ofk_warp_t, float32 x2); EPI_CONSIST the consistency byte through maps.om and, when epi.valid is set, the
// valid byte through maps.ov (a uint8 map then); no vector store.
template <bool MASKS, int EPI, int NP, int NB, int LA, int PW>
__global__ void __launch_bounds__((NCW + PW) * 32, 2) c3_ws_kernel(const __grid_constant__ Maps maps,
                                                               const float2* __restrict__ G,
                                                               const uint8_t* __restrict__ Gm, float sign,
                                                               int H, int W, unsigned tiles_x, unsigned tiles_per_frame,
                                                               unsigned total_tiles, uint64_t negzero2,
                                                               const EpiArgs<EPI> epi) {
    // a P stage is released one tile late (its rows double as the staging buffer of the output store)
    static_assert(NP >= NB + LA + 1, "P stages must outlive the box pipeline and the output store");
    using SM = Smem<NP, NB>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SM& sm = *reinterpret_cast<SM*>(smem_raw);   // no static shared memory in this kernel: the window starts aligned
    if (smem_u32(smem_raw) & 127u) __trap();
    const unsigned tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
    const unsigned first = blockIdx.x, stride = gridDim.x;
    if (first >= total_tiles) return;
    const unsigned T = (total_tiles - first + stride - 1) / stride;
    constexpr uint32_t P_BYTES = TS * TS * 8 + (MASKS ? TS * TS : 0);
    constexpr uint32_t B_BYTES = BH * BW * 8 + (MASKS ? BH * BMW : 0);

    if (tid == 0) {
        for (int k = 0; k < NP; ++k) { mbar_init(&sm.pfull[k], 1); mbar_init(&sm.pempty[k], NCW); }
        for (int k = 0; k < NB; ++k) { mbar_init(&sm.bfull[k], 1); mbar_init(&sm.bempty[k], NCW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (PW == 2 && wrp == NCW + 1) {
        // -------------------------------------------------------------------------------------------- P loader warp
        // Streams the pointwise tiles into the ring of P stages as fast as stages are released: independent of the
        // box pipeline, so neither the box warp nor the consumers ever wait for a P request to be issued.
        if (lane == 0) {
            const int tiles_y = (int)(tiles_per_frame / tiles_x);
            TileIter pit;
            pit.init(first, stride, (int)tiles_x, tiles_y);
            unsigned ps_i = 0, ps_ph = 0;
            for (unsigned i = 0; i < T; ++i) {
                const int tx0 = pit.tx * TS, ty0 = pit.ty * TS, n = pit.n;
                pit.advance((int)tiles_x, tiles_y);
                if (i >= NP) mbar_wait(&sm.pempty[ps_i], ps_ph ^ 1);
                mbar_expect_tx(&sm.pfull[ps_i], P_BYTES);
                tma_load_3d(sm.ps[ps_i].p, &maps.p, &sm.pfull[ps_i], tx0, ty0, n);
                if (MASKS) tma_load_3d(sm.ps[ps_i].pm, &maps.pm, &sm.pfull[ps_i], tx0, ty0, n);
                if (++ps_i == NP) { ps_i = 0; ps_ph ^= 1; }
            }
        }
        return;
    }
    if (wrp == NCW) {
        // ------------------------------------------------------------------------------------------ producer warp
        const int tiles_y = (int)(tiles_per_frame / tiles_x);
        TileIter pit, bit;   // cursors of the P loads and of the box preparation
        pit.init(first, stride, (int)tiles_x, tiles_y);
        bit = pit;
        unsigned ps_i = 0, ps_ph = 0;      // P stage / phase of the next P load
        auto issue_p = [&](bool wait_empty) {   // lane 0 only; tiles are issued in order
            const int tx0 = pit.tx * TS, ty0 = pit.ty * TS, n = pit.n;
            pit.advance((int)tiles_x, tiles_y);
            if (wait_empty) mbar_wait(&sm.pempty[ps_i], ps_ph ^ 1);
            mbar_expect_tx(&sm.pfull[ps_i], P_BYTES);
            tma_load_3d(sm.ps[ps_i].p, &maps.p, &sm.pfull[ps_i], tx0, ty0, n);
            if (MASKS) tma_load_3d(sm.ps[ps_i].pm, &maps.pm, &sm.pfull[ps_i], tx0, ty0, n);
            if (++ps_i == NP) { ps_i = 0; ps_ph ^= 1; }
        };
        if (PW == 1 && lane == 0)
            for (unsigned k = 0; k < (unsigned)LA && k < T; ++k) issue_p(false);
        unsigned s = 0, s_ph = 0, b = 0, b_ph = 0;
        for (unsigned i = 0; i < T; ++i) {
            const int tx0 = bit.tx * TS, ty0 = bit.ty * TS, n = bit.n;
            bit.advance((int)tiles_x, tiles_y);
            if (lane == 0) OFK_TR(i, 0);
            mbar_wait(&sm.pfull[s], s_ph);
            if (lane == 0) OFK_TR(i, 1);
            // Sample positions on a 4 x 4 grid over the tile (corners included): exact bounding box for affine fields, an
            // estimate otherwise (consumers verify per pixel). One shared-memory load per lane, four integer warp
            // reductions (REDUX): the producer's serial time per tile is what paces the whole pipeline.
            int x0, x1, y0, y1;
            {
                const int r = (int)(((lane >> 2) & 3) * 31 + 1) / 3, c = (int)((lane & 3) * 31 + 1) / 3;   // 0, 10, 21, 31
                const int x = tx0 + c, y = ty0 + r;
                int fx0 = 0x7fffffff, fx1 = -0x7fffffff, fy0 = 0x7fffffff, fy1 = -0x7fffffff;
                if (x < W && y < H) {
                    const float2 v = sm.ps[s].p[r * TS + c];
                    const float lim = 60000.f;
                    const float X = fminf(fmaxf(__fmaf_rn(sign, v.x, (float)x), -lim), lim);
                    const float Y = fminf(fmaxf(__fmaf_rn(sign, v.y, (float)y), -lim), lim);
                    fx0 = fx1 = __float2int_rd(X);
                    fy0 = fy1 = __float2int_rd(Y);
                }
                x0 = __reduce_min_sync(0xffffffffu, fx0); x1 = __reduce_max_sync(0xffffffffu, fx1);
                y0 = __reduce_min_sync(0xffffffffu, fy0); y1 = __reduce_max_sync(0xffffffffu, fy1);
            }
            if (lane == 0) {
                // integer tap range, clamped to the taps that can contribute: ix in [-1, W-1], iy in [-1, H-1]
                x0 = max(-1, min(W - 1, x0)); x1 = max(-1, min(W - 1, x1));
                y0 = max(-1, min(H - 1, y0)); y1 = max(-1, min(H - 1, y1));
                // centre the needed range [x0, x1 + 1] in the box (spare margin on both sides for curved flows)
                const int needw = x1 + 2 - x0, needh = y1 + 2 - y0;
                int vx0 = x0 - max(0, (BW - needw) / 2);
                vx0 &= ~1;                                   // 16-byte aligned box start (float2 elements)
                const int by0 = y0 - max(0, (BH - needh) / 2);
                const int mx0 = vx0 & ~15;
                OFK_TR(i, 2);
                if (i >= NB) mbar_wait(&sm.bempty[b], b_ph ^ 1);
                OFK_TR(i, 3);
                sm.binfo[b][0] = make_int4(vx0, vx0 - mx0, by0, 0);
                sm.binfo[b][1] = make_int4(tx0, ty0, n, 0);
                mbar_expect_tx(&sm.bfull[b], B_BYTES);
                tma_load_3d(sm.bs[b].v, &maps.gb, &sm.bfull[b], vx0, by0, n);
                if (MASKS) tma_load_3d(sm.bs[b].m, &maps.gmb, &sm.bfull[b], mx0, by0, n);
                OFK_TR(i, 4);
                if (PW == 1 && i + LA < T) issue_p(i + LA >= NP);
                OFK_TR(i, 5);
            }
            __syncwarp();
            if (++s == NP) { s = 0; s_ph ^= 1; }
            if (++b == NB) { b = 0; b_ph ^= 1; }
        }
        return;
    }

    // ---------------------------------------------------------------------------------------------- consumer warps
    const uint64_t one2 = pack2(1.0f, 1.0f);
    unsigned s = 0, s_ph = 0, b = 0, b_ph = 0;
    int prev_s = -1;
    for (unsigned i = 0; i < T; ++i) {
        if (lane == 0 && wrp == 0) OFK_TR(i, 8);
        if (lane == 0 && wrp == 7) OFK_TR(i, 12);
        mbar_wait(&sm.bfull[b], b_ph);
        mbar_wait(&sm.pfull[s], s_ph);
        if (lane == 0 && wrp == 0) OFK_TR(i, 9);
        if (lane == 0 && wrp == 7) OFK_TR(i, 13);
        const int4 info = sm.binfo[b][0], tile = sm.binfo[b][1];
        typename SM::PStage& ps = sm.ps[s];
        const typename SM::BStage& bs = sm.bs[b];
        const int tx0 = tile.x, ty0 = tile.y, n = tile.z;
        const float xg = (float)(tx0 + (int)lane);
        float2* prow = ps.p + ((int)wrp * 4 * TS + lane);      // this thread's pixels: prow[j * TS], in place
        uint8_t* mrow = ps.pm + ((int)wrp * 4 * TS + lane);

        uint64_t p[4];
        unsigned pm[4];
        int dx[4], dy[4], fa[4], fb[4];
        bool ok = true;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            p[j] = *reinterpret_cast<const uint64_t*>(prow + j * TS);
            pm[j] = MASKS ? mrow[j * TS] : 1u;
            const float2 pv = unpack2(p[j]);
            const float X = __fmaf_rn(sign, pv.x, xg), Y = __fmaf_rn(sign, pv.y, (float)(ty0 + (int)wrp * 4 + j));
            int ix, iy;
            quant(X, ix, fa[j]);
            quant(Y, iy, fb[j]);
            dx[j] = ix - info.x;
            dy[j] = iy - info.z;
            // Covered by the box? Everything else is decided per pixel. No range test is needed for the fast quantiser:
            // it is exact for |X| < 2^17, and beyond that (or for NaN / Inf) the integer it produces is far outside
            // [-2^16, 2^16], so such a pixel can never pass the box test (frames are smaller than 32768).
            ok = ok && (unsigned)dx[j] < (unsigned)(BW - 1) && (unsigned)dy[j] < (unsigned)(BH - 1);
        }
        unsigned vb[4];   // valid bytes of the consistency epilogue
        if (__all_sync(0xffffffffu, ok)) {
            uint64_t t[4][4];
            unsigned m[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint64_t* v = reinterpret_cast<const uint64_t*>(bs.v) + (dy[j] * BW + dx[j]);
                t[j][0] = v[0]; t[j][1] = v[1]; t[j][2] = v[BW]; t[j][3] = v[BW + 1];
                if (MASKS) {
                    const uint8_t* mm = bs.m + (dy[j] * BMW + dx[j] + info.y);
                    m[j][0] = mm[0]; m[j][1] = mm[1]; m[j][2] = mm[BMW]; m[j][3] = mm[BMW + 1];
                }
            }
            // validity and a reduction over every tap first: once they are known all taps of this warp have left the
            // box and the stage can be handed back to the producer while the blend is still running
            unsigned strict[4], dep = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const unsigned a = fa[j], bb = fb[j];
                const unsigned ha = min(a, 1u), hb = min(bb, 1u);      // 1 where the right / lower taps have weight
                if (MASKS) {
                    strict[j] = m[j][0] & (m[j][1] | ~ha) & (m[j][2] | ~hb) & (m[j][3] | ~(ha & hb)) & pm[j];
                } else {
                    const int ix = dx[j] + info.x, iy = dy[j] + info.z;
                    strict[j] = (ix >= 0 && iy >= 0 && (ix + 1 < W || (a == 0 && ix < W)) &&
                                 (iy + 1 < H || (bb == 0 && iy < H))) ? 1u : 0u;
                }
                // every tap feeds the release below (bit 8, masked off when the validity byte is stored): the loads
                // may be issued in any order, so "the value loaded last" is not something the source can name
                strict[j] |= (unsigned)((t[j][0] | t[j][1] | t[j][2] | t[j][3]) >> 63) << 8;
                dep |= strict[j];
            }
            dep = __reduce_or_sync(0xffffffffu, dep);
            if (lane == 0) mbar_arrive_after(&sm.bempty[b], dep, &sm.sink[wrp]);
            if (lane == 0 && wrp == 0) OFK_TR(i, 10);
            if (lane == 0 && wrp == 7) OFK_TR(i, 14);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const unsigned a = fa[j], bb = fb[j];
                const float ffa = (float)a * (1.0f / 32.0f), ffb = (float)bb * (1.0f / 32.0f);
                const uint64_t fa2 = pack2(ffa, ffa), fb2 = pack2(ffb, ffb);
                const uint64_t na2 = add2(one2, fa2 ^ 0x8000000080000000ull), nb2 = add2(one2, fb2 ^ 0x8000000080000000ull);
                uint64_t accv = mul2_nofuse(t[j][0], mul2(na2, nb2), negzero2);
                accv = add2(accv, mul2_nofuse(t[j][1], mul2(fa2, nb2), negzero2));
                accv = add2(accv, mul2_nofuse(t[j][2], mul2(na2, fb2), negzero2));
                accv = add2(accv, mul2_nofuse(t[j][3], mul2(fa2, fb2), negzero2));
                epilogue<EPI>(prow, mrow, j, p[j], accv, strict[j] & 1u, vb[j], epi);
            }
            stage_valid<EPI>(prow, vb, epi);
        } else {
            // Some pixel of this warp is not covered by the box. Along the frame border that is the rule (the box is
            // clamped to the frame): those pixels sample nothing but the zero border. Pixels that need taps from inside
            // the frame (discontinuous or noisy flow, estimate too small) send the warp to the out-of-line path.
            bool need_global = false;
            const int bx = cold_value(info.x), by = cold_value(info.z);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int ix = dx[j] + bx, iy = dy[j] + by;
                const bool inbox = (unsigned)dx[j] < (unsigned)(BW - 1) && (unsigned)dy[j] < (unsigned)(BH - 1);
                need_global = need_global || !(inbox || ix < -1 || iy < -1 || ix >= W || iy >= H);
            }
            if (__any_sync(0xffffffffu, need_global)) {
                if constexpr (EPI == EPI_CONSIST)
                    mixed_rows<MASKS, EPI, SM>(&ps, &bs, &sm.bempty[b], &sm.sink[wrp], info, tile, G, Gm, sign, H, W,
                                               negzero2, epi);
                else
                    mixed_rows<MASKS, EPI, SM>(&ps, &bs, &sm.bempty[b], &sm.sink[wrp], info, tile, G, Gm, sign, H, W,
                                               negzero2);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float2 pv = unpack2(p[j]);
                    const bool inbox = (unsigned)dx[j] < (unsigned)(BW - 1) && (unsigned)dy[j] < (unsigned)(BH - 1);
                    float su = 0.f, sv = 0.f;
                    unsigned strict = 0;
                    if (inbox) {
                        const float2* v = bs.v + (dy[j] * BW + dx[j]);
                        const float2 t00 = v[0], t01 = v[1], t10 = v[BW], t11 = v[BW + 1];
                        const int a = fa[j], bb = fb[j];
                        const unsigned za = a == 0, zb = bb == 0;
                        if (MASKS) {
                            const uint8_t* mm = bs.m + (dy[j] * BMW + dx[j] + info.y);
                            strict = mm[0] & (mm[1] | za) & (mm[BMW] | zb) & (mm[BMW + 1] | za | zb);
                        } else {
                            const int ix = dx[j] + info.x, iy = dy[j] + info.z;
                            strict = (ix >= 0 && iy >= 0 && (ix + 1 < W || (za && ix < W)) && (iy + 1 < H || (zb && iy < H))) ? 1u : 0u;
                        }
                        const float ffa = (float)a * (1.0f / 32.0f), ffb = (float)bb * (1.0f / 32.0f);
                        const float na = 1.0f - ffa, nb = 1.0f - ffb;
                        const float f00 = __fmul_rn(na, nb), f01 = __fmul_rn(ffa, nb), f10 = __fmul_rn(na, ffb),
                                    f11 = __fmul_rn(ffa, ffb);
                        su = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t00.x, f00), __fmul_rn(t01.x, f01)),
                                                 __fmul_rn(t10.x, f10)), __fmul_rn(t11.x, f11));
                        sv = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(t00.y, f00), __fmul_rn(t01.y, f01)),
                                                 __fmul_rn(t10.y, f10)), __fmul_rn(t11.y, f11));
                    }
                    if constexpr (EPI == EPI_CONSIST) {
                        vb[j] = pm[j] & strict & 1u;
                        mrow[j * TS] = (uint8_t)(vb[j] & fb_consistent(pv.x, pv.y, su, sv, epi.a1, epi.a2));
                    } else {
                        prow[j * TS] = EPI == EPI_COMPOSE ? make_float2(__fadd_rn(pv.x, su), __fadd_rn(pv.y, sv))
                                                          : make_float2(su, sv);
                        mrow[j * TS] = (uint8_t)(pm[j] & strict & 1u);
                    }
                }
                stage_valid<EPI>(prow, vb, epi);
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.bempty[b]);
            }
        }
        // the warp's 4 result rows go out as two bulk tensor stores (clipped at the frame border by the hardware)
        fence_async_smem();
        __syncwarp();
        // (issued under elect.sync: the compiler moves the operands to uniform registers without a waterfall loop)
        const int u_tx = tx0, u_ty = ty0 + (int)wrp * 4, u_n = n;
        const uint32_t u_src = smem_u32(ps.p + (int)wrp * 4 * TS), u_srcm = smem_u32(ps.pm + (int)wrp * 4 * TS);
        bool vec_store = true;
        if constexpr (EPI == EPI_CONSIST) vec_store = epi.valid != nullptr;
        if (elect_one()) {
            if (vec_store) tma_store_3d_u(&maps.ov, u_src, u_tx, u_ty, u_n);
            tma_store_3d_u(&maps.om, u_srcm, u_tx, u_ty, u_n);
            bulk_commit();
            if (prev_s >= 0) {
                bulk_wait_read<1>();                 // the previous tile's rows have been read out of shared memory
                mbar_arrive(&sm.pempty[prev_s]);
            }
        }
        if (lane == 0 && wrp == 0) OFK_TR(i, 11);
        if (lane == 0 && wrp == 7) OFK_TR(i, 15);
        prev_s = (int)s;
        if (++s == NP) { s = 0; s_ph ^= 1; }
        if (++b == NB) { b = 0; b_ph ^= 1; }
    }
    if (elect_one()) bulk_wait_all();   // the lane that committed the groups
}

// ------------------------------------------------------------------------------------------------ zero tests
__device__ __forceinline__ bool nz(float c, float thr) { return thr > 0.f ? !(c < thr && c > -thr) : (c != 0.f); }

// flags[n*2 + k] = 1 if a sparse sample of operand k of frame n (A: k = 0, B: k = 1) shows a non-zero vector on a
// valid pixel. One CTA per frame; PROBE_SAMPLES pixels per operand, spread over the frame.
constexpr int PROBE_SAMPLES = 2048;
__global__ void __launch_bounds__(256) c3_probe_nonzero(const float2* __restrict__ A, const uint8_t* __restrict__ Am,
                                                        const float2* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                        float thr, int* __restrict__ flags, size_t frame,
                                                        int stride /* flags per frame: 2, or 1 when B == NULL */) {
    const int n = blockIdx.x;
    const size_t base = (size_t)n * frame;
    const size_t step = frame / PROBE_SAMPLES > 0 ? frame / PROBE_SAMPLES : 1;
    bool a = false, b = false;
    for (size_t k = threadIdx.x; k < PROBE_SAMPLES; k += blockDim.x) {
        const size_t i = k * step;
        if (i >= frame) break;
        const float2 va = __ldg(A + base + i);
        a = a || ((Am == nullptr || Am[base + i]) && (nz(va.x, thr) || nz(va.y, thr)));
        if (B != nullptr) {
            const float2 vb = __ldg(B + base + i);
            b = b || ((Bm == nullptr || Bm[base + i]) && (nz(vb.x, thr) || nz(vb.y, thr)));
        }
    }
    const int fa = __syncthreads_or(a), fb = __syncthreads_or(b);
    if (threadIdx.x == 0) {
        flags[n * stride + 0] = fa ? 1 : 0;
        if (B != nullptr) flags[n * stride + 1] = fb ? 1 : 0;
    }
}

// Complete scan of the operands the probe left undecided (flag still 0); CTAs of decided frames exit at once.
__global__ void __launch_bounds__(256) c3_scan_nonzero(const float2* __restrict__ A, const uint8_t* __restrict__ Am,
                                                       const float2* __restrict__ B, const uint8_t* __restrict__ Bm,
                                                       float thr, int* __restrict__ flags, size_t frame, int stride) {
    const int n = blockIdx.y;
    // flags were written by the previous kernel
    const bool need_a = flags[n * stride + 0] == 0, need_b = B != nullptr && flags[n * stride + 1] == 0;
    if (!need_a && !need_b) return;
    const size_t base = (size_t)n * frame;
    bool a = false, b = false;
    const size_t step = (size_t)gridDim.x * blockDim.x;
    for (size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < frame; i0 += 4 * step) {
        // four independent loads per operand in flight
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const size_t i = i0 + k * step;
            if (i >= frame) break;
            if (need_a) {
                const float2 v = __ldg(A + base + i);
                a = a || ((Am == nullptr || Am[base + i]) && (nz(v.x, thr) || nz(v.y, thr)));
            }
            if (need_b) {
                const float2 v = __ldg(B + base + i);
                b = b || ((Bm == nullptr || Bm[base + i]) && (nz(v.x, thr) || nz(v.y, thr)));
            }
        }
    }
    const int fa = __syncthreads_or(a), fb = __syncthreads_or(b);
    if (threadIdx.x == 0) {
        if (fa) atomicOr(&flags[n * stride + 0], 1);
        if (fb) atomicOr(&flags[n * stride + 1], 1);
    }
}

// ------------------------------------------------------------------------------------------------ host side
constexpr int WS_NP = 5, WS_NB = 3, WS_LA = 1;   // 5 P stages, 3 box stages (LA only matters with a single producer warp)
constexpr int WS_PW = 2;                         // producer warps: box warp + P loader warp

}  // namespace c3ws

unsigned long long c3_ws_mixed_count() {
    unsigned long long v = 0;
    if (cudaMemcpyFromSymbol(&v, c3ws::g_mixed_warp_tiles, sizeof(v)) != cudaSuccess) cudaGetLastError();
    return v;
}

bool c3_ws_enabled() {
    static std::atomic<int> state{-1};
    if (state.load() < 0) {
        const char* e = getenv("OFK_C3_WS");
        state.store((e != nullptr && e[0] == '0') ? 0 : 1);
    }
    return state.load() == 1;
}

// The zero tests: flags[n] = {A_nonzero, B_nonzero} (combine3), or flags[n] = A_nonzero when B == NULL
// (ofk_nonzero_flags). 2 launches; the second is a no-op for frames the probe decided.
int launch_c3_zero_flags(const float* A, const uint8_t* Am, const float* B, const uint8_t* Bm, float thr, int* flags,
                         int N, int H, int W, cudaStream_t st) {
    const size_t frame = (size_t)H * W;
    const int stride = B != nullptr ? 2 : 1;
    c3ws::c3_probe_nonzero<<<N, 256, 0, st>>>((const float2*)A, Am, (const float2*)B, Bm, thr, flags, frame, stride);
    OFK_LAUNCHED();
    int bx = (int)((frame + 256 * 16 - 1) / (256 * 16));
    if (bx > 64) bx = 64;
    c3ws::c3_scan_nonzero<<<dim3(bx, N), 256, 0, st>>>((const float2*)A, Am, (const float2*)B, Bm, thr, flags, frame,
                                                        stride);
    OFK_LAUNCHED();
    return OFK_OK;
}

namespace c3ws {
// Maps of the pointwise operand, its mask and the gathered operand and its mask; false if an operand does not fit the
// TMA kernel (caller uses the rows kernel)
static bool input_maps(Maps& maps, const float* P, const uint8_t* Pm, const float* G, const uint8_t* Gm, int N, int H,
                       int W) {
    if ((Pm == nullptr) != (Gm == nullptr)) return false;
    if (W % 16 != 0) return false;   // 16-byte row pitch of the uint8 tensors (output mask always, input masks if given)
    if (H >= 32768 || W >= 32768) return false;
    if (!make_map3(&maps.p, P, 8, W, H, N, TS, TS) || !make_map3(&maps.gb, G, 8, W, H, N, BW, BH)) return false;
    if (Pm != nullptr) {
        if (!make_map3(&maps.pm, Pm, 1, W, H, N, TS, TS) || !make_map3(&maps.gmb, Gm, 1, W, H, N, BMW, BH)) return false;
    } else {
        maps.pm = maps.gmb = maps.p;
    }
    return true;
}

template <bool MK, int EPI>
static int launch_ws(const Maps& maps, const float* G, const uint8_t* Gm, float sign, int N, int H, int W,
                     const EpiArgs<EPI>& epi, cudaStream_t st) {
    const unsigned tx = (W + TS - 1) / TS, ty = (H + TS - 1) / TS;
    if ((double)tx * ty * N >= 4.0e9) return 0;
    const unsigned total = tx * ty * (unsigned)N;
    unsigned grid = (unsigned)sm_count() * 2;
    if (grid > total) grid = total;
    grid = ws::cap_ctas(grid);
    const size_t smem = sizeof(Smem<WS_NP, WS_NB>);
    static std::atomic<bool> attr_done_dev[64];   // the attribute is per device; racing threads set it twice
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    std::atomic<bool>& attr_done = attr_done_dev[dev];
    if (!attr_done) {
        if (cudaFuncSetAttribute(c3_ws_kernel<MK, EPI, WS_NP, WS_NB, WS_LA, WS_PW>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return 0;
        }
        attr_done = true;
    }
    c3_ws_kernel<MK, EPI, WS_NP, WS_NB, WS_LA, WS_PW><<<grid, (NCW + WS_PW) * 32, smem, st>>>(
        maps, (const float2*)G, Gm, sign, H, W, tx, tx * ty, total, 0x8000000080000000ull, epi);
    OFK_LAUNCHED();
    return 1;
}
}  // namespace c3ws

// Returns 1 if the kernel was launched, 0 if the configuration is not eligible (caller uses the rows kernel),
// negative OFK_E* on error. P/G are the pointwise / gathered operands, sign = -1 ('t') or +1 ('s').
int launch_combine3_ws(const float* P, const uint8_t* Pm, const float* G, const uint8_t* Gm, float sign, bool add,
                       float* out, uint8_t* omask, int N, int H, int W, cudaStream_t st) {
    using namespace c3ws;
    Maps maps;
    if (!input_maps(maps, P, Pm, G, Gm, N, H, W) || !make_map3(&maps.ov, out, 8, W, H, N, TS, 4) ||
        !make_map3(&maps.om, omask, 1, W, H, N, TS, 4))
        return 0;
    const EpiArgs<EPI_COMPOSE> compose{};
    const EpiArgs<EPI_SAMPLE> sample{};
    if (Pm != nullptr) return add ? launch_ws<true>(maps, G, Gm, sign, N, H, W, compose, st)
                                  : launch_ws<true>(maps, G, Gm, sign, N, H, W, sample, st);
    return add ? launch_ws<false>(maps, G, Gm, sign, N, H, W, compose, st)
               : launch_ws<false>(maps, G, Gm, sign, N, H, W, sample, st);
}

// The consistency check of ofk_consistency through the TMA kernel: P = F, G = G, out / out_valid uint8 [N,H,W]
// (out_valid may be NULL). Returns as launch_combine3_ws.
int launch_consistency_ws(const float* F, const uint8_t* Fm, const float* G, const uint8_t* Gm, float sign, float a1,
                          float a2, uint8_t* out, uint8_t* out_valid, int N, int H, int W, cudaStream_t st) {
    using namespace c3ws;
    Maps maps;
    if (!input_maps(maps, F, Fm, G, Gm, N, H, W) || !make_map3(&maps.om, out, 1, W, H, N, TS, 4)) return 0;
    if (out_valid != nullptr) {
        if (!make_map3(&maps.ov, out_valid, 1, W, H, N, TS, 4)) return 0;
    } else {
        maps.ov = maps.om;   // not used
    }
    EpiArgs<EPI_CONSIST> epi;
    epi.a1 = a1;
    epi.a2 = a2;
    epi.valid = out_valid;
    return Fm != nullptr ? launch_ws<true>(maps, G, Gm, sign, N, H, W, epi, st)
                         : launch_ws<false>(maps, G, Gm, sign, N, H, W, epi, st);
}

}  // namespace ofk
