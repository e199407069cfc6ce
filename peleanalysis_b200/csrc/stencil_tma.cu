// stencil_tma.cu -- the hot stencil kernels as a persistent, TMA-staged shared-memory pipeline for sm_100a.
//
// Work item = (tile, variable); a tile = rows [y0,y0+ny) x planes [z0,z0+nz) of one box, full x extent, swept along z
// (2.5-D blocking).  Because a tile spans whole rows, the (ny+2) rows of one z-plane -- y halo and x ghosts included --
// are ONE contiguous, 16-byte aligned run in the box's slab, so a plane is staged with a single cp.async.bulk (TMA,
// SASS UBLKCP) that completes on an mbarrier.  Faces with a neighbour link (PaNbrFace) are staged straight from the
// neighbour box -- this rank's slab or a peer GPU's over NVLink: a z-ghost plane is one bulk copy from the
// neighbour's plane, a y-ghost row one row copy, an x-ghost column one 8-byte cp.async (LDGSTS) per row.
//
// The kernel is PERSISTENT: the grid is 2 CTAs per SM, each CTA draws work items from a global ticket counter (SMs do
// not all see the same HBM bandwidth, so a static split would wait for the slowest) and the S-stage ring of planes
// runs continuously across item boundaries -- the producer warp is already streaming the next
// tile while the consumers finish the current one, so there is no per-tile pipeline fill / drain and the descriptor
// loads of the next tile are off the consumers' critical path (the tile record travels through the ring with the
// tile's first plane).  Eight consumer warps read each plane from shared memory (128-bit LDS for the centre pair and
// the y neighbours, warp shuffles for the x neighbours), keep the z-1 / z / z+1 centre values in a register queue, and
// hand stages back to the producer through a second mbarrier -- no __syncthreads in the steady state.
// Arithmetic is the reference's expression order with separate IEEE mul/add (-fmad=false): bit-exact.
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>

#include "kernels.cuh"
#include "stencil_dev.cuh"

namespace pa {

namespace {

constexpr int MAX_STAGES = 16;
// Two CTA shapes (template parameter CW = consumer warps; + 1 producer warp each):
//   CW = 8,  2 CTAs/SM, 2 x-pairs per consumer thread per plane : the bandwidth-bound modes (two independent rings per SM)
//   CW = 16, 1 CTA/SM,  1 x-pair  per consumer thread per plane : the FP64-heavy flame-normal modes -- the same 16 consumer
//            warps per SM, but half the per-thread state and a 112-register budget (9 warps are allocated as 10, which
//            caps the 2-CTA shape at 96 registers and made the normal epilogue spill)
//   CW = 4 / 2 : tiles of small boxes (at most 256 / 128 x-pairs per plane, e.g. 32^3 / 16^3 boxes).  In the big shapes such
//            a tile would leave half / three quarters of the consumer threads idle while they still execute every
//            instruction; here the CTA is as wide as the tile and more CTAs (3-6) share an SM, so more tiles are in flight
constexpr int TILE_ITEMS = 512;                       // x-pairs per tile plane of the two big shapes: CW * 32 * ITEMS
template <int CW, bool HEAVY> struct Shape {
    static constexpr int NI = CW >= 16 ? 1 : 2;                                           // x-pairs per consumer thread
    static constexpr int CAP = CW * 32 * NI;                                              // x-pairs per tile plane
    // CTAs per SM; HEAVY = the flame-normal modes, which want ~112 registers
    static constexpr int PER_SM = CW >= 16 ? 1 : CW == 8 ? 2 : CW == 4 ? (HEAVY ? 3 : 4) : (HEAVY ? 5 : 6);
};
constexpr int MAX_TILE_ROWS = 30;                     // rows per tile: as many as MAX_ITEMS * CONSUMER_THREADS x-pairs allow, up to this
constexpr int XG_LANES = 30;                          // producer lanes 1 .. 30 fetch the x ghosts: (side, row) cells lane-1 and lane-1+30
constexpr int STATIC_SMEM = 10 * 1024 + 256;          // upper bound of the static shared memory below (10112 bytes)


template <int MODE> struct ModeTraits;
template <> struct ModeTraits<MODE_GRAD> { static constexpr int NIN = 1, NOUT = 4; };
template <> struct ModeTraits<MODE_GRAD3> { static constexpr int NIN = 1, NOUT = 3; };
template <> struct ModeTraits<MODE_NORMAL> { static constexpr int NIN = 1, NOUT = 3; };
template <> struct ModeTraits<MODE_DIV> { static constexpr int NIN = 3, NOUT = 1; };
template <> struct ModeTraits<MODE_NORMAL_S> { static constexpr int NIN = 1, NOUT = 3; };

// what the consumers need to know about a work item; written by producer lane 0 into the ring slot of the item's
// first plane, so it is protected by that stage's full / empty barriers like the plane data itself
struct TileRec {
    PaTile t;
    int v;                   // variable (blockIdx.y of the non-persistent formulation)
    int links;               // bit f set: face f has a neighbour link
    PaBoxDev bx;
    PaLayDev li, lo;
};

// per-item flags (one register)
enum : unsigned {
    F_ACTIVE = 1u, F_TWO = 2u,           // item exists; its second cell is a valid cell (not the x-hi ghost of an odd row)
    F_EDGE_LO = 4u, F_EDGE_HI = 8u,      // x-1 / x+2 must come from shared memory (lane or row boundary), not from a shuffle
    F_XLO_LINK = 16u, F_XHI_LINK = 32u,  // first / last pair of a row whose x ghost comes from a linked neighbour (xg_s)
    F_XM_RAW = 64u, F_XP_RAW = 128u,     // MODE_NORMAL_S: that neighbour is a materialised ghost (already progress space)
    F_YM_RAW = 256u, F_YP_RAW = 512u, F_CY_RAW = 1024u,   // ... same for the y neighbours / the pair's second cell
    F_ROW_SHIFT = 16
};

// PLAIN = true: the flame normal through the plain IEEE operators (sqrt(), six divisions) instead of normal_pair() -- the
// form the library falls back to should the device self-test of the branch-free forms ever report a differing bit
template <int MODE, int CW, bool PLAIN>
__global__ void __launch_bounds__((CW + 1) * 32, Shape<CW, MODE == MODE_NORMAL || MODE == MODE_NORMAL_S>::PER_SM) k_stencil_tma(const PaTile* __restrict__ tiles, int ntiles, int nwork, GridArgs ga,
                                                            StencilExtra ex, int stage_doubles /* per input component, multiple of 16 */,
                                                            int S /* ring depth in planes */,
                                                            unsigned long long* __restrict__ ticket, unsigned long long ticket_base,
                                                            int psleep /* ns between the producer's polls of an empty barrier; 0 = spin */) {
    constexpr int NIN = ModeTraits<MODE>::NIN;
    constexpr int NOUT = ModeTraits<MODE>::NOUT;
    constexpr bool XS = (MODE == MODE_NORMAL_S);
    constexpr int CONSUMER_WARPS = CW, CONSUMER_THREADS = CW * 32, MAX_ITEMS = Shape<CW, false>::NI;
    PA_DYN_SMEM(smem_raw);
    double* sm = reinterpret_cast<double*>(smem_raw);                 // [S][NIN][stage_doubles]
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
    __shared__ __align__(16) double xg_s[MAX_STAGES][2][32];          // x ghosts of linked x faces: [stage][lo/hi][row]
    __shared__ __align__(16) TileRec rec_s[MAX_STAGES];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long stage_stride = (long long)NIN * stage_doubles;

    if (threadIdx.x == 0) {
        // a stage is full when the TMA bytes have landed (lane 0's arrive.expect_tx) and every x-ghost lane has arrived
        for (int s = 0; s < S; ++s) { mbar_init(&full_bar[s], 1u + XG_LANES); mbar_init(&empty_bar[s], CONSUMER_WARPS); }
#ifndef PA_HOST_EMULATION
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
    }
    __syncthreads();

    const bool hint_ld = (psleep & (1 << 30)) != 0, hint_st = (psleep & (1 << 29)) != 0;   // PA_TMA_L2HINT bits 0 / 1 (launch_mode)
    psleep &= 0xffff;
#define TMA_LOAD(d_, s_, n_, b_) do { if (hint_ld) tma_load_1d_hint(d_, s_, n_, b_, l2pol); else tma_load_1d(d_, s_, n_, b_); } while (0)
    if (warp == CONSUMER_WARPS) {
        // ===================================== producer warp =====================================
        // lane 0 drives the TMA ring; lanes 1 .. 2*ny each own one x-ghost cell (side, row) per plane of a linked x face;
        // lanes without such a cell just arrive, so the full barrier's arrival count is the same for every tile.
        if (lane > XG_LANES) return;
        const uint64_t l2pol = hint_ld ? l2_policy_evict_last() : 0;
        int stage = 0;
        uint32_t ephase = 1;                            // parity that lets the first pass through the ring go without waiting
        for (;;) {
            // next work item: the counter is never reset -- the host advances ticket_base by (nwork + grid) per launch,
            // exactly what the CTAs of one launch draw in total (every CTA overdraws once, then stops)
            unsigned long long tk = 0;
            if (lane == 0) tk = atomicAdd(ticket, 1ULL) - ticket_base;
            tk = __shfl_sync(0x7fffffffu, tk, 0);
            if (tk >= (unsigned long long)nwork) {
                // end marker for the consumers: an empty record in one more ring slot
                if (psleep) mbar_wait_sleep(&empty_bar[stage], ephase, (unsigned)psleep); else mbar_wait(&empty_bar[stage], ephase);
                if (lane == 0) { rec_s[stage].t.lev = -1; mbar_arrive(&full_bar[stage]); }
                else cp_async_arrive_noinc(&full_bar[stage]);
                break;
            }
            const int wi = (int)tk;
            const int v = wi / ntiles;
            const PaTile t = tiles[wi - v * ntiles];
            const LevArgs& L = ga.L[t.lev];
            const PaBoxDev bx = L.boxes[t.box];
            const PaLayDev li = L.lay_in[t.box];
            const PaNbr nb = L.nbr[t.box];
            const int c0 = L.in_comp + (MODE == MODE_DIV ? 0 : v);
            const int rows = t.ny + 2, nplanes = t.nz + 2;
            const uint32_t row_bytes = (uint32_t)li.P * 8u, plane_bytes = (uint32_t)rows * row_bytes;
            // per linked face: address of the neighbour element matching (row 0 of the padded block, plane 0, x pad 0) of
            // component c0, and the component stride of the slab it lives in.  neighbour-relative cell = own-relative + rel
            auto link_src = [&](int face, long long& cs) -> const double* {
                const PaNbrFace F = nb.f[face];
                cs = 0;
                if (F.nb < 0) return nullptr;
                const PaPeerSlab ps = L.peers[F.rank];
                const PaLayDev ln = L.lay_in[F.nb];
                cs = ps.cs;
                return ps.base + (long long)c0 * ps.cs + ln.off + (long long)(F.rel[2] + ln.ng) * ln.PS + (long long)(F.rel[1] + ln.ng) * ln.P + F.rel[0];
            };
            const double* own = L.in + (MODE == MODE_DIV ? 0 : (long long)v * L.cs_in) + li.off + (long long)li.ng * li.PS + (long long)li.ng * li.P;
            // lane 0: sources of the linked y / z faces; lanes 1..: source of this lane's x-ghost cell at plane 0
            long long cs_ylo = 0, cs_zlo = 0, cs_yhi = 0, cs_zhi = 0;
            const double *s_ylo = nullptr, *s_zlo = nullptr, *s_yhi = nullptr, *s_zhi = nullptr;
            const double* xsrc[2] = {nullptr, nullptr};            // this lane's (up to two) x-ghost cells at plane 0
            double* xdst[2] = {nullptr, nullptr};                  // ... and where they go inside stage 0's xg_s block
            if (lane == 0) {
                s_ylo = link_src(1, cs_ylo);                       // rel[0] == 0 for y and z faces: rows are x-aligned
                s_zlo = link_src(2, cs_zlo);
                s_yhi = link_src(4, cs_yhi);
                s_zhi = link_src(5, cs_zhi);
            } else {
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int idx = lane - 1 + XG_LANES * k;
                    const int side = idx / t.ny, xr = idx - side * t.ny;   // side 0 = x-lo, 1 = x-hi
                    if (side < 2) {
                        long long cs;
                        const double* s0 = link_src(side ? 3 : 0, cs);
                        // own-relative ghost cell (gi, y0 + xr, z0 - 1 + p): gi = -1 (lo) or nx (hi)
                        if (s0) {
                            xsrc[k] = s0 + (long long)(t.z0 - 1) * li.PS + (long long)(t.y0 + xr) * li.P + ((side ? bx.n[0] : -1) + li.ng + li.xoff);
                            xdst[k] = &xg_s[0][side][xr];
                        }
                    }
                }
            }
            const int nyb = bx.n[1], nzb = bx.n[2];
            for (int p = 0; p < nplanes; ++p) {
                if (psleep) mbar_wait_sleep(&empty_bar[stage], ephase, (unsigned)psleep); else mbar_wait(&empty_bar[stage], ephase);
                if (lane == 0) {
                    if (p == 0) {                                  // the tile record rides with the tile's first plane
                        TileRec& R = rec_s[stage];
                        R.t = t; R.v = v; R.bx = bx; R.li = li; R.lo = L.lay_out[t.box];
                        int lk = 0;
#pragma unroll
                        for (int f = 0; f < 6; ++f) lk |= (nb.f[f].nb >= 0) ? (1 << f) : 0;
                        R.links = lk;
                    }
                    mbar_expect_tx(&full_bar[stage], plane_bytes * NIN);
                    const int z = t.z0 - 1 + p;
                    const double* zs = (z < 0) ? s_zlo : (z >= nzb ? s_zhi : nullptr);
                    const long long zcs = (z < 0) ? cs_zlo : cs_zhi;
#pragma unroll
                    for (int c = 0; c < NIN; ++c) {
                        double* dst = sm + (long long)stage * stage_stride + (long long)c * stage_doubles;
                        if (zs) {
                            TMA_LOAD(dst, zs + (long long)c * zcs + (long long)z * li.PS + (long long)(t.y0 - 1) * li.P, plane_bytes, &full_bar[stage]);
                            continue;
                        }
                        int r0 = t.y0 - 1, r1 = t.y0 + t.ny;             // first / last staged row (box-relative)
                        if (r0 < 0 && s_ylo) {
                            TMA_LOAD(dst, s_ylo + (long long)c * cs_ylo + (long long)z * li.PS - li.P, row_bytes, &full_bar[stage]);
                            r0 = 0;
                        }
                        if (r1 >= nyb && s_yhi) {
                            TMA_LOAD(dst + (long long)(rows - 1) * li.P, s_yhi + (long long)c * cs_yhi + (long long)z * li.PS + (long long)nyb * li.P,
                                        row_bytes, &full_bar[stage]);
                            r1 = nyb - 1;
                        }
                        TMA_LOAD(dst + (long long)(r0 - (t.y0 - 1)) * li.P, own + (long long)c * L.cs_in + (long long)z * li.PS + (long long)r0 * li.P,
                                    (uint32_t)(r1 - r0 + 1) * row_bytes, &full_bar[stage]);
                    }
                } else {
                    if (xsrc[0]) cp_async_8(xdst[0] + stage * 64, xsrc[0] + (long long)p * li.PS);
                    if (xsrc[1]) cp_async_8(xdst[1] + stage * 64, xsrc[1] + (long long)p * li.PS);
                    cp_async_arrive_noinc(&full_bar[stage]);
                }
                if (++stage == S) { stage = 0; ephase ^= 1u; }
            }
        }
        return;
    }

    // ===================================== consumer warps =====================================
    int sc = 0;                    // stage of the plane being received
    uint32_t fphase = 0;
    auto wait_full = [&](int st, uint32_t ph) { mbar_wait(&full_bar[st], ph); };
    auto arrive_empty = [&](int st) { mbar_arrive(&empty_bar[st]); };
    const double pmin = ex.pmin, pinv = ex.inv;
    auto prog = [&](double sv) { return (sv - pmin) * pinv; };          // curvature.cpp:316-320

    for (;;) {
        // ---- plane 0 of the tile (z = z0-1) and the tile record ----
        wait_full(sc, fphase);
        const TileRec& R = rec_s[sc];
        const PaTile t = R.t;
        if (t.lev < 0) break;                          // end marker
        const int v = R.v, links = R.links;
        const int nx = R.bx.n[0], nyb = R.bx.n[1], nzb = R.bx.n[2];
        const int P = R.li.P;
        const int lo_P = R.lo.P;
        const long long lo_PS = R.lo.PS;
        const LevArgs& L = ga.L[t.lev];
        const double dxi = L.dxi[0], dyi = L.dxi[1], dzi = L.dxi[2];
        const long long cs_out = L.cs_out;
        double* __restrict__ out0 = L.out + (long long)v * NOUT * cs_out;
        const int nq = (nx + 1) >> 1;
        const int items = nq * t.ny;                   // <= MAX_ITEMS * CONSUMER_THREADS by tile construction
        const int xbase = R.li.ng + R.li.xoff;         // even
        const int nplanes = t.nz + 2;
        // MODE_NORMAL_S: staged values are the raw scalar S wherever they come from valid cells (own or a linked
        // neighbour's) and already-normalised progress values where they are this box's materialised ghost cells
        const bool z0_raw = XS && t.z0 == 0 && !(links & 4);
        const bool zl_raw = XS && t.z0 + t.nz == nzb && !(links & 32);

        int soff[MAX_ITEMS];                           // centre pair inside one component block of a stage
        unsigned fl[MAX_ITEMS];
        long long oo[MAX_ITEMS];                       // output element offset of the item in the plane being written
        double2 cm[MAX_ITEMS], c0[MAX_ITEMS];          // register queue: centre pairs of planes p-2 and p-1
        long long pi[MAX_ITEMS];                       // MODE_DIV threshold: the item's cell in the input layout (progress variable)
        const int li_PS = R.li.PS;
#pragma unroll
        for (int it = 0; it < MAX_ITEMS; ++it) {
            const int w = threadIdx.x + it * CONSUMER_THREADS;
            const bool active = w < items;
            const int q = active ? (w % nq) : 0;
            const int r = active ? (w / nq) : 0;
            soff[it] = (r + 1) * P + xbase + 2 * q;
            oo[it] = R.lo.off + (long long)(t.z0 + R.lo.ng) * lo_PS + (long long)(t.y0 + r + R.lo.ng) * lo_P + (2 * q + R.lo.ng + R.lo.xoff);
            unsigned f = (unsigned)r << F_ROW_SHIFT;
            if (active) f |= F_ACTIVE;
            if (2 * q + 1 < nx) f |= F_TWO;
            if (lane == 0 || q == 0) f |= F_EDGE_LO;
            if (lane == 31 || q == nq - 1 || !active || w + 1 >= items) f |= F_EDGE_HI;
            if (q == 0 && (links & 1)) f |= F_XLO_LINK;
            if (q == nq - 1 && (links & 8)) f |= F_XHI_LINK;
            if (XS) {
                if (q == 0 && !(links & 1)) f |= F_XM_RAW;
                if (q == nq - 1 && !(links & 8)) f |= (nx & 1) ? F_CY_RAW : F_XP_RAW;
                if (t.y0 + r == 0 && !(links & 2)) f |= F_YM_RAW;
                if (t.y0 + r == nyb - 1 && !(links & 16)) f |= F_YP_RAW;
            }
            fl[it] = f;
            pi[it] = R.li.off + (long long)(t.z0 + R.li.ng) * li_PS + (long long)(t.y0 + r + R.li.ng) * P + (2 * q + xbase);
            cm[it] = c0[it] = make_double2(0., 0.);
        }
        // centre pair of the z-derivative component of a freshly landed plane (MODE_DIV: n_z), fixed up so that the
        // register queue always holds final values: linked x-hi ghost of an odd row, progress normalisation
        auto load_centre = [&](int st, int it, bool plane_raw) -> double2 {
            const double* Sq = sm + (long long)st * stage_stride + (MODE == MODE_DIV ? 2 * stage_doubles : 0) + soff[it];
            double2 c = lds2(Sq);
            if (MODE != MODE_DIV) {
                if ((fl[it] & F_XHI_LINK) && (nx & 1)) c.y = xg_s[st][1][fl[it] >> F_ROW_SHIFT];    // the pair's second cell IS the ghost
                if (XS && !plane_raw) { c.x = prog(c.x); if (!(fl[it] & F_CY_RAW)) c.y = prog(c.y); }
            }
            return c;
        };
#pragma unroll
        for (int it = 0; it < MAX_ITEMS; ++it) c0[it] = load_centre(sc, it, z0_raw);
        int sp = sc;                                   // stage of plane p-1
        if (++sc == S) { sc = 0; fphase ^= 1u; }

        // per-tile invariants of the epilogues (kernel parameters indexed by the level: one load per tile, not per plane)
        double* const cout_base = XS ? ex.cout[t.lev] : nullptr;
        double* const aux_base = (MODE == MODE_NORMAL || MODE == MODE_NORMAL_S) ? ex.aux[t.lev] : nullptr;
        const long long cg = (MODE == MODE_NORMAL || MODE == MODE_NORMAL_S) ? ex.cs_aux[t.lev] : 0;
        const double* const prog_base = (MODE == MODE_DIV && ex.do_threshold) ? ex.prog[t.lev] : nullptr;
        const bool xlo_link = (links & 1) != 0, xhi_link_even = (links & 8) != 0 && !(nx & 1);

        for (int p = 1; p < nplanes; ++p) {
            wait_full(sc, fphase);
            const double* Sp = sm + (long long)sp * stage_stride;
            const bool last_raw = zl_raw && p == nplanes - 1;
#pragma unroll
            for (int it = 0; it < MAX_ITEMS; ++it) {
                const unsigned f = fl[it];
                const double2 cp = load_centre(sc, it, last_raw);
                if (p >= 2) {
                    // ---- finish plane p-1: in-plane derivatives from its stage, z derivative from the register queue ----
                    // Everything up to the stores is branch-free (selects, not divergent branches: lanes 0 and 31 of every
                    // warp are "edge" lanes), so the two items' chains can be scheduled side by side.
                    const double* Sc = Sp + soff[it];
                    const int row = (int)(f >> F_ROW_SHIFT);
                    double2 c = c0[it];
                    if (MODE == MODE_DIV) {
                        c = lds2(Sc);                                      // n_x centre pair
                        if ((f & F_XHI_LINK) && (nx & 1)) c.y = xg_s[sp][1][row];
                    }
                    // x neighbours: from the adjacent lanes when they hold the same row, else from shared memory -- the
                    // staged row (own cells / materialised ghost) or, on a linked x face, the neighbour's column in xg_s
                    double xm = __shfl_up_sync(0xffffffffu, c.y, 1);
                    double xp = __shfl_down_sync(0xffffffffu, c.x, 1);
                    double el = Sc[-1], eh = Sc[2];
                    if (xlo_link) { const double gl = xg_s[sp][0][row]; el = (f & F_XLO_LINK) ? gl : el; }
                    if (xhi_link_even) { const double gh = xg_s[sp][1][row]; eh = (f & F_XHI_LINK) ? gh : eh; }
                    if (XS) {
                        const double pl = prog(el), ph = prog(eh);
                        el = (f & F_XM_RAW) ? el : pl;
                        eh = (f & F_XP_RAW) ? eh : ph;
                    }
                    xm = (f & F_EDGE_LO) ? el : xm;
                    xp = (f & F_EDGE_HI) ? eh : xp;
                    const double ax = cdiff(dxi, xm, c.x, c.y);
                    const double ay = cdiff(dxi, c.x, c.y, xp);
                    double bx0, by0;
                    if (MODE != MODE_DIV) {
                        double2 ym = lds2(Sc - P), yp = lds2(Sc + P);
                        if (XS) {
                            const double a0 = prog(ym.x), a1 = prog(ym.y), b0 = prog(yp.x), b1 = prog(yp.y);
                            ym.x = (f & F_YM_RAW) ? ym.x : a0; ym.y = (f & F_YM_RAW) ? ym.y : a1;
                            yp.x = (f & F_YP_RAW) ? yp.x : b0; yp.y = (f & F_YP_RAW) ? yp.y : b1;
                        }
                        bx0 = cdiff(dyi, ym.x, c.x, yp.x);
                        by0 = cdiff(dyi, ym.y, c.y, yp.y);
                    } else {
                        const double* Sy = Sc + stage_doubles;              // component 1 (n_y)
                        const double2 cy = lds2(Sy), ym = lds2(Sy - P), yp = lds2(Sy + P);
                        bx0 = cdiff(dyi, ym.x, cy.x, yp.x);
                        by0 = cdiff(dyi, ym.y, cy.y, yp.y);
                    }
                    const double g0 = cdiff(dzi, cm[it].x, c0[it].x, cp.x);
                    const double g1 = cdiff(dzi, cm[it].y, c0[it].y, cp.y);
                    const bool act = (f & F_ACTIVE) != 0, two = (f & F_TWO) != 0;
                    const long long o = oo[it];
                    double r0[4], r1[4];
                    if (MODE == MODE_GRAD) {
                        r0[0] = ax; r0[1] = bx0; r0[2] = g0; r0[3] = sqrt(ax * ax + bx0 * bx0 + g0 * g0);
                        r1[0] = ay; r1[1] = by0; r1[2] = g1; r1[3] = sqrt(ay * ay + by0 * by0 + g1 * g1);
                    } else if (MODE == MODE_GRAD3) {
                        r0[0] = ax; r0[1] = bx0; r0[2] = g0;
                        r1[0] = ay; r1[1] = by0; r1[2] = g1;
                    } else if (MODE == MODE_NORMAL || MODE == MODE_NORMAL_S) {
                        if (PLAIN) {
                            const double n0 = -fmax(1e-14, sqrt(ax * ax + bx0 * bx0 + g0 * g0));
                            const double n1 = -fmax(1e-14, sqrt(ay * ay + by0 * by0 + g1 * g1));
                            r0[0] = ax / n0; r0[1] = bx0 / n0; r0[2] = g0 / n0;
                            r1[0] = ay / n1; r1[1] = by0 / n1; r1[2] = g1 / n1;
                        } else {
                            normal_pair(ax, bx0, g0, ay, by0, g1, r0, r1);
                        }
                    } else {
                        r0[0] = 0.5 * (((0.0 + ax) + bx0) + g0);
                        r1[0] = 0.5 * (((0.0 + ay) + by0) + g1);
                    }
                    if (act) {
                        if (XS) {                                            // Progress of plane p-1 (curvature.cpp:310-321)
                            double* pc = cout_base + o;
                            if (two) { if (hint_st) stg2_cs(pc, c.x, c.y); else stg2(pc, c.x, c.y); } else pc[0] = c.x;
                        }
                        if ((MODE == MODE_NORMAL || MODE == MODE_NORMAL_S) && aux_base) {
                            double* g = aux_base + o;
                            if (two) { stg2(g, ax, ay); stg2(g + cg, bx0, by0); stg2(g + 2 * cg, g0, g1); }
                            else { g[0] = ax; g[cg] = bx0; g[2 * cg] = g0; }
                        }
                        if (MODE == MODE_DIV && prog_base) {
                            const double2 pc = *reinterpret_cast<const double2*>(prog_base + pi[it]);
                            if (pc.x < ex.threshold || pc.x > 1.0 - ex.threshold) r0[0] = 0.0;
                            if (pc.y < ex.threshold || pc.y > 1.0 - ex.threshold) r1[0] = 0.0;
                        }
                        double* po = out0 + o;
#pragma unroll
                        for (int m = 0; m < NOUT; ++m) {
                            if (two) { if (hint_st) stg2_cs(po, r0[m], r1[m]); else stg2(po, r0[m], r1[m]); } else po[0] = r0[m];
                            po += cs_out;
                        }
                    }
                    oo[it] += lo_PS;
                    if (MODE == MODE_DIV) pi[it] += li_PS;
                }
                cm[it] = c0[it];
                c0[it] = cp;
            }
            // this warp no longer needs plane p-1
            __syncwarp();
            if (lane == 0) arrive_empty(sp);
            sp = sc;
            if (++sc == S) { sc = 0; fphase ^= 1u; }
        }
        // ... nor the tile's last plane
        __syncwarp();
        if (lane == 0) arrive_empty(sp);
    }
}

// host-side launch bookkeeping below (ticket table, per-kernel shared-memory attribute, cached device properties) is shared
// by all host threads of the process; launches from different threads (each on its own stream) serialise on this mutex
std::mutex g_launch_mutex;
// work-item ticket counters, one per stream (launches on one stream are ordered, so they can share a counter that is
// never reset; kernels on different streams may overlap and must not)
struct Ticket { unsigned long long* dev = nullptr; unsigned long long base = 0; };
std::map<std::pair<int, cudaStream_t>, Ticket> g_tickets;         // (device, stream): host threads may drive several GPUs
int g_stage_cap = 0;
size_t g_inflight_bytes = 0;

template <int MODE, int CW, bool PLAIN>
cudaError_t launch_mode(const PaTile* tiles, int ntiles, int stage_doubles, const GridArgs& ga, const StencilExtra& ex,
                        int nvar, cudaStream_t st) {
    constexpr int NIN = ModeTraits<MODE>::NIN;
    constexpr bool HEAVY = MODE == MODE_NORMAL || MODE == MODE_NORMAL_S;
    constexpr int PER_SM = Shape<CW, HEAVY>::PER_SM;
    constexpr int THREADS = (CW + 1) * 32;
    std::lock_guard<std::mutex> lock(g_launch_mutex);
    const size_t stage_bytes = (size_t)NIN * stage_doubles * sizeof(double);
    // Ring depth.  The consumers hold two planes (p-1 and p); the rest of the ring is data in flight.  Measured on B200
    // (config 2): ~40 KB in flight per SM (~6 MB chip-wide = bandwidth x latency) is the optimum -- a deeper
    // ring is SLOWER (the read stream runs far ahead of the write stream and the two fight for DRAM pages / L2).
    if (g_inflight_bytes == 0) { const char* e = getenv("PA_TMA_INFLIGHT_KB"); g_inflight_bytes = (size_t)(e ? std::max(1, atoi(e)) : 20) * 1024; }
    const size_t inflight = g_inflight_bytes * 2 / PER_SM;
    constexpr size_t STATIC = STATIC_SMEM;
    const size_t budget = (size_t)(227 * 1024) / PER_SM - STATIC - 1024, budget1 = 227 * 1024 - STATIC - 1024;
    int S = 2 + (int)((inflight + stage_bytes - 1) / stage_bytes), per_sm = PER_SM;
    if ((size_t)S * stage_bytes > budget) S = (int)(budget / stage_bytes);
    if (S < 3) { S = std::min(4, (int)(budget1 / stage_bytes)); per_sm = 1; }
    if (S < 3) return cudaErrorInvalidConfiguration;
    if (S > MAX_STAGES) S = MAX_STAGES;
    if (g_stage_cap == 0) { const char* e = getenv("PA_TMA_STAGES"); g_stage_cap = e ? std::max(3, atoi(e)) : MAX_STAGES; }
    if (S > g_stage_cap) S = g_stage_cap;
    const size_t smem = (size_t)S * stage_bytes;
    int dev = 0;
    { cudaError_t e = cudaGetDevice(&dev); if (e != cudaSuccess) return e; }
    static std::map<int, size_t> configured;                          // per device: the attribute lives in the device's context
    if (smem > configured[dev]) {
        cudaError_t e = cudaFuncSetAttribute(k_stencil_tma<MODE, CW, PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[dev] = smem;
    }
    cudaError_t esm = cudaSuccess;
    const int num_sms = stencil_num_sms(&esm);
    if (esm != cudaSuccess) return esm;
    const long long nwork = (long long)ntiles * nvar;
    const int grid = (int)std::min<long long>(nwork, (long long)num_sms * per_sm);
    Ticket& T = g_tickets[std::make_pair(dev, st)];
    if (!T.dev) {
        cudaError_t e = dev_alloc((void**)&T.dev, sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaMemset(T.dev, 0, sizeof(unsigned long long));
        if (e != cudaSuccess) return e;
    }
    const char* eps = getenv("PA_TMA_PSLEEP");
    // L2 eviction hints (bit 0: evict_last on the staged loads, bit 1: streaming stores).  Measured on a B200
    // (profiles/r02_ab_l2_hints.txt): the bandwidth-bound gradient modes gain 2.5 % with both (config 2: 92.4 -> 95.0 % of the
    // roofline, DRAM reads 7.04 -> 6.48 GB for 5.6 GB of input: fewer halo rows shared by neighbouring tiles are fetched twice).  The
    // curvature step as a whole does not (6.58 -> 6.65 ms) -- but kernel by kernel (ncu launch list, end of round 2,
    // profiles/r02_ablate_normal_f3.txt) the flame-normal pass loses (3.73 -> 3.87 ms) and the read-dominated divergence wins
    // (2.22 -> 2.13 ms, DRAM reads 11.2 -> 10.4 GB), so the divergence takes the hints and the flame-normal pass does not.
    const char* eh = getenv("PA_TMA_L2HINT");
    const int hints = eh ? atoi(eh) : ((MODE == MODE_GRAD || MODE == MODE_GRAD3 || MODE == MODE_DIV) ? 3 : 0);
    const int psleep = (eps ? std::min(std::max(0, atoi(eps)), 0xffff) : 0) | ((hints & 1) << 30) | (((hints >> 1) & 1) << 29);
    PA_LAUNCH(grid, THREADS, smem, st, k_stencil_tma<MODE, CW, PLAIN>)(tiles, ntiles, (int)nwork, ga, ex, stage_doubles, S, T.dev, T.base, psleep);
    T.base += (unsigned long long)nwork + (unsigned long long)grid;
    return cudaGetLastError();
}

// which modes run in the 16-consumer-warp shape: bit m = mode m (PA_TMA_CW16 overrides; default: the two flame-normal modes)
int g_cw16_mask = -1;
// Flame-normal arithmetic of the TMA kernel: 0 = branch-free forms (normal_pair), 1 = plain IEEE operators, -1 = not decided.
// PA_NORMAL_MATH=fast|plain forces one; otherwise ("auto") the first flame-normal launch of the process runs the device
// self-test once (2^20 operand sets, well under a millisecond) and the branch-free forms are used only if not one result
// bit differs from sqrt() / division on THIS device and driver -- the transcribed sequences depend on the MUFU seeds.
int g_normal_plain = -1;
std::mutex g_cfg_mutex;                               // guards the lazily decided settings (host threads may launch concurrently)
int decide_normal_math(cudaStream_t st) {
    std::lock_guard<std::mutex> lock(g_cfg_mutex);
    if (g_normal_plain >= 0) return g_normal_plain;
    const char* e = getenv("PA_NORMAL_MATH");
    if (e && !strcmp(e, "plain")) return g_normal_plain = 1;
    if (e && !strcmp(e, "fast")) return g_normal_plain = 0;
    unsigned long long bad = 0;
    const cudaError_t ce = selftest_math(1LL << 20, 0x9A5EEDULL, &bad, st);
    g_normal_plain = (ce != cudaSuccess || bad != 0) ? 1 : 0;
    if (g_normal_plain)
        fprintf(stderr, "[pelestencil_b200] branch-free flame-normal self-test: %llu differing results (%s) -- using the plain IEEE operators\n",
                bad, cudaGetErrorString(ce));
    return g_normal_plain;
}
// PA_TMA_SMALL=0 switches the small-tile shapes (4 / 2 consumer warps) off (read at every launch: the tests flip it)
template <int MODE, bool PLAIN>
cudaError_t launch_cw(int cw, const PaTile* tiles, int ntiles, int stage_doubles, const GridArgs& ga, const StencilExtra& ex,
                       int nvar, cudaStream_t st) {
    switch (cw) {
        case 2: return launch_mode<MODE, 2, PLAIN>(tiles, ntiles, stage_doubles, ga, ex, nvar, st);
        case 4: return launch_mode<MODE, 4, PLAIN>(tiles, ntiles, stage_doubles, ga, ex, nvar, st);
        case 16: return launch_mode<MODE, 16, PLAIN>(tiles, ntiles, stage_doubles, ga, ex, nvar, st);
        default: return launch_mode<MODE, 8, PLAIN>(tiles, ntiles, stage_doubles, ga, ex, nvar, st);
    }
}
template <int MODE>
cudaError_t launch_shape(const PaTile* tiles, int ntiles, int stage_doubles, int max_items, const GridArgs& ga, const StencilExtra& ex,
                         int nvar, cudaStream_t st) {
    int mask16;
    {
        std::lock_guard<std::mutex> lock(g_cfg_mutex);
        if (g_cw16_mask < 0) { const char* e = getenv("PA_TMA_CW16"); g_cw16_mask = e ? atoi(e) : ((1 << MODE_NORMAL) | (1 << MODE_NORMAL_S)); }
        mask16 = g_cw16_mask;
    }
    const char* es = getenv("PA_TMA_SMALL");
    int cw = (mask16 & (1 << MODE)) ? 16 : 8;
    if (!(es && es[0] == '0') && max_items > 0) {
        if (max_items <= Shape<2, false>::CAP) cw = 2;
        else if (max_items <= Shape<4, false>::CAP) cw = 4;
    }
    if constexpr (MODE == MODE_NORMAL || MODE == MODE_NORMAL_S) {
        if (decide_normal_math(st)) return launch_cw<MODE, true>(cw, tiles, ntiles, stage_doubles, ga, ex, nvar, st);
    }
    return launch_cw<MODE, false>(cw, tiles, ntiles, stage_doubles, ga, ex, nvar, st);
}

// ---- device self-test of the branch-free math against the plain operators --------------------------------------
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {          // splitmix64 finaliser
    z += 0x9E3779B97F4A7C15ULL; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL; z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__device__ __forceinline__ bool same_bits(double a, double b) {
    return (a != a && b != b) || __double_as_longlong(a) == __double_as_longlong(b);
}
// a double with a random sign / mantissa and an exponent drawn uniformly from [e0, e1]; every 16th mantissa is 0 or all ones
__device__ __forceinline__ double rnd_double(unsigned long long r, int e0, int e1, bool neg_ok) {
    unsigned long long m = r & 0x000FFFFFFFFFFFFFULL;
    const unsigned sel = (unsigned)(r >> 52) & 15u;
    if (sel == 0) m = 0; else if (sel == 1) m = 0x000FFFFFFFFFFFFFULL;
    const unsigned long long e = (unsigned long long)(e0 + (int)((r >> 20) % (unsigned long long)(e1 - e0 + 1)));
    const unsigned long long sg = neg_ok ? (r >> 63) : 0ULL;
    return __longlong_as_double((long long)((sg << 63) | (e << 52) | m));
}
__global__ void k_selftest_math(long long n, unsigned long long seed, unsigned long long* __restrict__ bad) {
    unsigned long long local = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long r0 = mix64(seed + 4ULL * (unsigned long long)i), r1 = mix64(r0), r2 = mix64(r1), r3 = mix64(r2);
        // sqrt_fast on its whole range [2^-970, inf), and on near-squares (the hard rounding cases)
        double x = rnd_double(r0, 0x035, 0x7fe, false);
        if (sqrt_fast_ok(x) && !same_bits(sqrt_fast(x), sqrt(x))) ++local;
        const double y = rnd_double(r1, 0x200, 0x5ff, false);
        x = __longlong_as_double(__double_as_longlong(y * y) + (long long)(r1 % 5ULL) - 2);
        if (sqrt_fast_ok(x) && !same_bits(sqrt_fast(x), sqrt(x))) ++local;
        // rcp_fast on the divisors the flame normal produces: 1e-14 <= |n| <= 2^513 (and the fast-path guard agrees)
        const double d = rnd_double(r2, 0x3d0, 0x600, true);
        if (!rcp_fast_ok(d) || !same_bits(rcp_fast(d), __drcp_rn(d))) ++local;
        // the whole flame-normal pair against the plain formula, components spread over 2^-1074 .. 2^600, zeros included
        double g[6];
        unsigned long long r = r3;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            r = mix64(r);
            const unsigned cls = (unsigned)(r >> 40) & 15u;
            if (cls == 0) g[k] = (r >> 63) ? -0.0 : 0.0;
            else if (cls == 1) g[k] = rnd_double(r, 0x000, 0x0d0, true);             // denormals and tiny normals
            else if (cls == 2) g[k] = rnd_double(r, 0x600, 0x658, true);             // G.G overflows for the largest
            else if (cls < 6) g[k] = rnd_double(r, 0x3c0, 0x3e0, true);              // around the 1e-14 clamp
            else g[k] = rnd_double(r, 0x3f0 - (int)((r >> 8) & 63u), 0x410, true);   // ordinary gradients, mixed magnitudes
        }
        double q0[3], q1[3];
        normal_pair(g[0], g[1], g[2], g[3], g[4], g[5], q0, q1);
        {   // the quad form of the fused curvature kernel on the same operands (cells 0 / 1 as they are, 2 / 3 permuted)
            const double qx[4] = {g[0], g[3], g[1], g[5]}, qy[4] = {g[1], g[4], g[2], g[3]}, qz[4] = {g[2], g[5], g[0], g[4]};
            double m0[4], m1[4], m2[4];
            normal_quad(qx, qy, qz, m0, m1, m2);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double nn = -fmax(1e-14, sqrt(qx[j] * qx[j] + qy[j] * qy[j] + qz[j] * qz[j]));
                if (!same_bits(m0[j], qx[j] / nn)) ++local;
                if (!same_bits(m1[j], qy[j] / nn)) ++local;
                if (!same_bits(m2[j], qz[j] / nn)) ++local;
            }
        }
        const double n0 = -fmax(1e-14, sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]));
        const double n1 = -fmax(1e-14, sqrt(g[3] * g[3] + g[4] * g[4] + g[5] * g[5]));
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (!same_bits(q0[k], g[k] / n0)) ++local;
            if (!same_bits(q1[k], g[3 + k] / n1)) ++local;
        }
    }
    if (local) atomicAdd(bad, local);
}

}  // namespace

cudaError_t selftest_math(long long n, unsigned long long seed, unsigned long long* bad_host, cudaStream_t st) {
    unsigned long long* d = nullptr;
    cudaError_t e = dev_alloc((void**)&d, sizeof(unsigned long long));
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(d, 0, sizeof(unsigned long long), st);
    int nsm = 0;
    if (e == cudaSuccess) nsm = stencil_num_sms(&e);
    if (e == cudaSuccess) { PA_LAUNCH(nsm * 8, 256, 0, st, k_selftest_math)(n, seed, d); ++g_launches; e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaMemcpyAsync(bad_host, d, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    dev_free(d);
    return e;
}

int stencil_tma_normal_math() { std::lock_guard<std::mutex> lock(g_cfg_mutex); return g_normal_plain; }
int stencil_decide_normal_math(cudaStream_t st) { return decide_normal_math(st); }
// SM count of the current device (cached per device)
int stencil_num_sms(cudaError_t* err) {
    static std::map<int, int> cache;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    int dev = 0;
    *err = cudaGetDevice(&dev);
    if (*err != cudaSuccess) return 0;
    auto it = cache.find(dev);
    if (it != cache.end()) return it->second;
    int n = 0;
    *err = cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (*err != cudaSuccess) return 0;
    cache[dev] = n;
    return n;
}
// the stream's work-item ticket counter for a persistent launch that draws `nwork` items with `grid` CTAs (every CTA
// overdraws once): returns the counter and the base the kernel subtracts, and advances the base
cudaError_t stencil_ticket(cudaStream_t st, unsigned long long nwork, int grid, unsigned long long** dev_out, unsigned long long* base_out) {
    std::lock_guard<std::mutex> lock(g_launch_mutex);
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    Ticket& T = g_tickets[std::make_pair(dev, st)];
    if (!T.dev) {
        e = dev_alloc((void**)&T.dev, sizeof(unsigned long long));
        if (e == cudaSuccess) e = cudaMemset(T.dev, 0, sizeof(unsigned long long));
        if (e != cudaSuccess) return e;
    }
    *dev_out = T.dev; *base_out = T.base;
    T.base += nwork + (unsigned long long)grid;
    return cudaSuccess;
}
void stencil_tma_release() {                          // pa_finalize: the per-stream ticket counters
    std::lock_guard<std::mutex> lock(g_launch_mutex);
    for (auto& kv : g_tickets) if (kv.second.dev) dev_free(kv.second.dev);
    g_tickets.clear();
}
int stencil_tma_tile_rows() { return MAX_TILE_ROWS; }
int stencil_tma_max_tile_rows() { return MAX_TILE_ROWS; }
// largest staged plane ((TY+2) rows x pitch) the pipeline accepts per input component (3 stages of 3 components must fit)
int stencil_tma_max_plane_doubles() { return (227 * 1024 - STATIC_SMEM - 1024) / (3 * 3 * 8); }

cudaError_t launch_stencil_tma(int mode, const PaTile* tiles, int ntiles, int max_plane_doubles, int max_items, const GridArgs& ga,
                               const StencilExtra& ex, int nvar, cudaStream_t st) {
    if (ntiles <= 0) return cudaSuccess;
    int stage_doubles = (max_plane_doubles + 15) & ~15;
    cudaError_t e;
    switch (mode) {
        case MODE_GRAD: e = launch_shape<MODE_GRAD>(tiles, ntiles, stage_doubles, max_items, ga, ex, nvar, st); break;
        case MODE_GRAD3: e = launch_shape<MODE_GRAD3>(tiles, ntiles, stage_doubles, max_items, ga, ex, nvar, st); break;
        case MODE_NORMAL: e = launch_shape<MODE_NORMAL>(tiles, ntiles, stage_doubles, max_items, ga, ex, nvar, st); break;
        case MODE_DIV: e = launch_shape<MODE_DIV>(tiles, ntiles, stage_doubles, max_items, ga, ex, nvar, st); break;
        case MODE_NORMAL_S: e = launch_shape<MODE_NORMAL_S>(tiles, ntiles, stage_doubles, max_items, ga, ex, nvar, st); break;
        default: return cudaErrorInvalidValue;
    }
    ++g_launches;
    return e;
}

}  // namespace pa
