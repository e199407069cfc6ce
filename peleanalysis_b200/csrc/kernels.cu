// kernels.cu -- hand-written sm_100a kernels of the ghost fill and the pointwise / simple stencil passes.
// Compiled with -fmad=false: every floating-point expression below is evaluated in the reference's order with
// separate IEEE multiplies and adds (the reference CPU build has no FMA), so results are bit-identical.
#include <atomic>
#include <cstdint>
#include <cstdlib>

#include "kernels.cuh"

namespace pa {

std::atomic<long long> g_launches{0};

#define PA_NAN __longlong_as_double(0x7ff8000000000000LL)

__device__ __forceinline__ int fdiv_dev(int a, int r) { return (a >= 0) ? a / r : -((-a + r - 1) / r); }

__device__ __forceinline__ long long cell_addr(const PaLayDev& y, int i, int j, int k) {
    // (i,j,k) relative to the valid box's low corner; ghosts are -ng..-1 and n..n+ng-1
    return y.off + (long long)(k + y.ng) * y.PS + (long long)(j + y.ng) * y.P + (i + y.ng + y.xoff);
}

template <class T>
__device__ __forceinline__ long long upper_idx(const T* a, long long lo, long long hi, long long c) {
    // largest r in [lo,hi) with a[r].start <= c
    while (hi - lo > 1) {
        long long mid = (lo + hi) >> 1;
        if (a[mid].start <= c) lo = mid; else hi = mid;
    }
    return lo;
}

static inline int grid_for(long long n, int block, int cap = 148 * 16) {
    long long g = (n + block - 1) / block;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

// ------------------------------------------------------------------------------------------------------------
// valid-region <-> host-ordered staging buffer (all local boxes of a level in one launch)
// ------------------------------------------------------------------------------------------------------------
template <bool TO_LAYOUT>
__global__ void k_valid_copy(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay,
                             const long long* __restrict__ host_off, int nboxes, long long ncells,
                             double* __restrict__ comp_base, double* __restrict__ staging) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        int lo = 0, hi = nboxes;
        while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (host_off[mid] <= c) lo = mid; else hi = mid; }
        const PaBoxDev b = boxes[lo];
        long long q = c - host_off[lo];
        int i = (int)(q % b.n[0]);
        long long r = q / b.n[0];
        int j = (int)(r % b.n[1]);
        int k = (int)(r / b.n[1]);
        long long a = cell_addr(lay[lo], i, j, k);
        if (TO_LAYOUT) comp_base[a] = staging[c]; else staging[c] = comp_base[a];
    }
}

cudaError_t launch_unpack_valid(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes,
                                long long ncells, const double* staging, double* comp_base, cudaStream_t st) {
    if (ncells <= 0) return cudaSuccess;
    PA_LAUNCH(grid_for(ncells, 256), 256, 0, st, k_valid_copy<true>)(boxes, lay, host_off, nboxes, ncells, comp_base, const_cast<double*>(staging));
    ++g_launches;
    return cudaGetLastError();
}
cudaError_t launch_pack_valid(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes,
                              long long ncells, const double* comp_base, double* staging, cudaStream_t st) {
    if (ncells <= 0) return cudaSuccess;
    PA_LAUNCH(grid_for(ncells, 256), 256, 0, st, k_valid_copy<false>)(boxes, lay, host_off, nboxes, ncells, const_cast<double*>(comp_base), staging);
    ++g_launches;
    return cudaGetLastError();
}

__global__ void k_fill(double* __restrict__ p, long long n, double v) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) p[c] = v;
}
cudaError_t launch_fill(double* p, long long n, double v, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    PA_LAUNCH(grid_for(n, 256), 256, 0, st, k_fill)(p, n, v);
    ++g_launches;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------------
// halo_gather: same-level + periodic ghost copies, one launch per level over the precomputed tag table.
// A tag whose source box lives on another rank reads the recv slab ([cell][comp] order) instead.
// ------------------------------------------------------------------------------------------------------------
__global__ void k_halo(const PaHaloTag* __restrict__ tags, int tag0, int tag1, long long cell0, long long cell1,
                       const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay, double* __restrict__ base,
                       long long cs, int ncomp, const double* __restrict__ recv, const PaPeerSlab* __restrict__ peers,
                       int comp0, int rank, GhostXform xf) {
    for (long long c = cell0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; c < cell1; c += (long long)gridDim.x * blockDim.x) {
        const PaHaloTag t = tags[upper_idx(tags, tag0, tag1, c)];
        long long q = c - t.start;
        int i = (int)(q % t.n[0]);
        long long r = q / t.n[0];
        int j = (int)(r % t.n[1]);
        int k = (int)(r / t.n[1]);
        const PaBoxDev db = boxes[t.dbox];
        const int di = t.dlo[0] + i, dj = t.dlo[1] + j, dk = t.dlo[2] + k;
        long long da = cell_addr(lay[t.dbox], di - db.lo[0], dj - db.lo[1], dk - db.lo[2]);
        if (t.sbox >= 0) {
            const PaBoxDev sb = boxes[t.sbox];
            long long sa = cell_addr(lay[t.sbox], di + t.shift[0] - sb.lo[0], dj + t.shift[1] - sb.lo[1], dk + t.shift[2] - sb.lo[2]);
            if (t.srank == rank) {
                for (int m = 0; m < ncomp; ++m) { double v = base[sa + m * cs]; base[da + m * cs] = xf.on ? (v - xf.pmin) * xf.inv : v; }
            } else {                                   // peer-owned link target: read its slab in place (NVLink)
                const PaPeerSlab ps = peers[t.srank];
                const double* s = ps.base + (long long)comp0 * ps.cs + sa;
                for (int m = 0; m < ncomp; ++m) { double v = s[m * ps.cs]; base[da + m * cs] = xf.on ? (v - xf.pmin) * xf.inv : v; }
            }
        } else {
            const double* s = recv + (t.rsrc + q) * ncomp;
            for (int m = 0; m < ncomp; ++m) { double v = s[m]; base[da + m * cs] = xf.on ? (v - xf.pmin) * xf.inv : v; }
        }
    }
}
cudaError_t launch_halo(const PaHaloTag* tags, int tag0, int tag1, long long cell0, long long cell1, const PaBoxDev* boxes,
                        const PaLayDev* lay, double* base, long long cs, int ncomp, const double* recv,
                        const PaPeerSlab* peers, int comp0, int rank, GhostXform xf, cudaStream_t st) {
    if (cell1 <= cell0 || tag1 <= tag0) return cudaSuccess;
    PA_LAUNCH(grid_for(cell1 - cell0, 256), 256, 0, st, k_halo)(tags, tag0, tag1, cell0, cell1, boxes, lay, base, cs, ncomp, recv, peers, comp0, rank, xf);
    ++g_launches;
    return cudaGetLastError();
}

// exchange pack: valid cells other ranks need (halo sources and coarse cells of their c-f registers) -> send slab,
// [cell][comp] order, all source levels in one launch.  Tags [tag0, tag1) enumerate cells [dense0, dense0+ncells).
__global__ void k_xpack(const PaPackTag* __restrict__ tags, long long tag0, long long tag1, long long dense0, long long ncells,
                        GridArgs ga, int ncomp, double* __restrict__ send) {
    for (long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x; w < ncells; w += (long long)gridDim.x * blockDim.x) {
        const long long c = w + dense0;
        long long lo = tag0, hi = tag1;
        while (hi - lo > 1) { long long mid = (lo + hi) >> 1; if (tags[mid].dense <= c) lo = mid; else hi = mid; }
        const PaPackTag t = tags[lo];
        const long long q = c - t.dense;
        int i = (int)(q % t.n[0]);
        long long r = q / t.n[0];
        int j = (int)(r % t.n[1]);
        int k = (int)(r / t.n[1]);
        const LevArgs& L = ga.L[t.slev];
        const PaBoxDev sb = L.boxes[t.sbox];
        long long sa = cell_addr(L.lay_in[t.sbox], t.slo[0] + i - sb.lo[0], t.slo[1] + j - sb.lo[1], t.slo[2] + k - sb.lo[2]);
        double* d = send + (t.start + q) * ncomp;
        for (int m = 0; m < ncomp; ++m) d[m] = L.in[sa + m * L.cs_in];
    }
}
cudaError_t launch_exchange_pack(const PaPackTag* tags, long long tag0, long long tag1, long long dense0, long long ncells,
                                 const GridArgs& ga, int ncomp, double* send, cudaStream_t st) {
    if (ncells <= 0 || tag1 <= tag0) return cudaSuccess;
    PA_LAUNCH(grid_for(ncells, 256), 256, 0, st, k_xpack)(tags, tag0, tag1, dense0, ncells, ga, ncomp, send);
    ++g_launches;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------------
// cf_bc_fill: every face ghost cell whose mask is > 0, all levels / boxes / faces in one launch.
//   physical face : Neumann copy or odd reflection                      (AMReX_MLLinOp_K.H:26-47)
//   coarse-fine   : bcval = tangential o3 interpolation of coarse data  (AMReX_InterpBndryData_3D_K.H:23-119)
//                   ghost = sum_{m>=1} coef[m]*phi(interior m) ; ghost += bcval*coef[0]   (AMReX_MLLinOp_K.H:48-68)
// Coarse values are gathered straight from the coarse level's valid cells through the precomputed index
// (no BndryRegister copy); an index of -1 means the reference's register cell was never filled (NaN).
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double xform(const GhostXform& xf, double v) { return xf.on ? (v - xf.pmin) * xf.inv : v; }

// value of a coarse register cell (pa_types.h: coarse gather offset table); `peers` / `pcomp` = the coarse level's peer slabs
// and the component's index inside the field (peer slabs are addressed from component 0)
__device__ __forceinline__ double crse_val(const long long* __restrict__ coff, long long e, const double* __restrict__ cbase,
                                           const double* __restrict__ recv, int ncomp, int comp, const GhostXform& xf,
                                           const PaPeerSlab* __restrict__ peers, int pcomp) {
    const long long a = coff[e];
    if (a >= 0) return xform(xf, cbase[a]);
    if (a == -1) return PA_NAN;
    if (a > -PA_CRSE_PEER_BASE) return xform(xf, recv[(-2 - a) * ncomp + comp]);
    const long long v = -a - PA_CRSE_PEER_BASE;
    const PaPeerSlab ps = peers[v >> PA_CRSE_PEER_SHIFT];
    return xform(xf, ps.base[(long long)pcomp * ps.cs + (v & ((1LL << PA_CRSE_PEER_SHIFT) - 1))]);
}

__global__ void __launch_bounds__(PA_FACE_CHUNK) k_bcfill(const PaFaceRec* __restrict__ recs, const int* __restrict__ rec_level,
                                                          const PaFaceBlock* __restrict__ blocks, const unsigned short* __restrict__ flags,
                                                          const long long* __restrict__ coff, GridArgs ga, int ncomp,
                                                          const double* __restrict__ recv, GhostXform xf) {
    const PaFaceBlock fb = blocks[blockIdx.x];
    const PaFaceRec R = recs[fb.rec];
    const int q = fb.cell0 + threadIdx.x;
    if (q >= R.n1 * R.n2) return;
    const unsigned fl = flags[R.start + q];
    if ((fl & 3u) == 0u) return;                                   // covered: the halo copy (or a neighbour link) owns this cell
    const int lev = rec_level[fb.rec];
    const LevArgs& L = ga.L[lev];
    const PaBoxDev bx = L.boxes[R.box];
    const PaLayDev ly = L.lay_in[R.box];
    const int a1 = q % R.n1, a2 = q / R.n1;
    const int d = R.face % 3;
    const int t1 = (d == 0) ? 1 : 0, t2 = (d == 2) ? 1 : 2;
    const int s = (R.face < 3) ? 1 : -1;
    int g[3];
    g[d] = (R.face < 3) ? -1 : bx.n[d];
    g[t1] = a1; g[t2] = a2;
    const long long ga_ = cell_addr(ly, g[0], g[1], g[2]);
    const long long sd = (d == 0) ? 1 : (d == 1) ? (long long)ly.P : (long long)ly.PS;
    for (int m = 0; m < ncomp; ++m) {
        double* p = L.out + ga_ + m * L.cs_in;
        if (R.kind == PA_FACE_NEUMANN) {
            *p = xform(xf, p[s * sd]);
        } else if (R.kind == PA_FACE_REFLECT_ODD) {
            *p = -xform(xf, p[s * sd]);
        } else {
            const LevArgs& LC = ga.L[lev - 1];
            const double* cbase = LC.in + m * LC.cs_in;
            const int r = R.ratio;
            const int j = bx.lo[t1] + a1, k = bx.lo[t2] + a2;
            const int jc = fdiv_dev(j, r), kc = fdiv_dev(k, r);
            const long long e0 = R.cidx + (long long)(kc - R.rlo2) * R.rn1 + (jc - R.rlo1);
#define CR(o1, o2) crse_val(coff, e0 + (long long)(o2) * R.rn1 + (o1), cbase, recv, ncomp, m, xf, LC.peers, LC.in_comp + m)
            const double c00 = CR(0, 0);
            int lo = PA_FLAG_NC(fl, 0) ? -1 : 0;
            int hi = PA_FLAG_NC(fl, 1) ? 1 : 0;
            double fac = (hi == lo + 1) ? 1.0 : 0.5;
            const double d1 = fac * (CR(hi, 0) - CR(lo, 0));
            const double d11 = (hi == lo + 2) ? 0.5 * (CR(1, 0) - 2. * c00 + CR(-1, 0)) : 0.;
            lo = PA_FLAG_NC(fl, 2) ? -1 : 0;
            hi = PA_FLAG_NC(fl, 3) ? 1 : 0;
            fac = (hi == lo + 1) ? 1.0 : 0.5;
            const double d2 = fac * (CR(0, hi) - CR(0, lo));
            const double d22 = (hi == lo + 2) ? 0.5 * (CR(0, 1) - 2. * c00 + CR(0, -1)) : 0.;
            const double d12 = (((fl >> 6) & 15u) == 15u)
                                   ? 0.25 * (CR(1, 1) - CR(-1, 1) + CR(-1, -1) - CR(1, -1)) : 0.0;
#undef CR
            const double x1 = -0.5 + (j - jc * r + 0.5) / r;
            const double x2 = -0.5 + (k - kc * r + 0.5) / r;
            const double bcval = c00 + x1 * d1 + (x1 * x1) * d11 + x2 * d2 + (x2 * x2) * d22 + x1 * x2 * d12;
            double tmp = 0.0;
            for (int mm = 1; mm < R.nx; ++mm) tmp += xform(xf, p[mm * s * sd]) * R.coef[mm];
            double v = tmp;
            v += bcval * R.coef[0];
            *p = v;
        }
    }
}
// ---- the default since round 2 (PA_BCFILL_V2=0 selects k_bcfill above, kept as the independent second route the tests compare;
// measured on a B200, profiles/r02_ab_variants.txt: grad on 16^3 boxes 0.983 -> 0.961 ms, curvature on 64^3 boxes 1.064 -> 1.036 ms,
// 128^3 boxes unchanged) ----
// Same arithmetic, different data path for the coarse values.  k_bcfill lets every ghost cell gather its (up to) nine
// coarse neighbours itself: nine offset-table loads and nine scattered 8-byte loads per cell, the same coarse cell fetched
// by up to nine threads (and r*r fine cells share a coarse cell): ncu shows 22-30 % DRAM utilisation at 8 useful bytes per
// 32-byte sector.  Here the block first stages the coarse register cells its chunk can touch -- the chunk's coarse footprint
// plus one cell all round -- in shared memory, each exactly once (row-contiguous, so coalesced for y / z faces), and the
// nine-point formula then reads shared memory.
constexpr int BCF_TILE = 640;        // coarse cells of a chunk's footprint incl. the one-cell rim (worst case: 128 rows of one cell, r = 2: 3 x 67)

__global__ void __launch_bounds__(PA_FACE_CHUNK) k_bcfill_v2(const PaFaceRec* __restrict__ recs, const int* __restrict__ rec_level,
                                                             const PaFaceBlock* __restrict__ blocks, const unsigned short* __restrict__ flags,
                                                             const long long* __restrict__ coff, GridArgs ga, int ncomp,
                                                             const double* __restrict__ recv, GhostXform xf) {
    __shared__ double cs[BCF_TILE];
    const PaFaceBlock fb = blocks[blockIdx.x];
    const PaFaceRec R = recs[fb.rec];
    const int ncell = R.n1 * R.n2;
    const int q = fb.cell0 + threadIdx.x;
    const bool inside = q < ncell;
    const unsigned fl = inside ? flags[R.start + q] : 0u;
    const bool active = inside && (fl & 3u) != 0u;                 // covered cells belong to the halo copy / a neighbour link
    const int lev = rec_level[fb.rec];
    const LevArgs& L = ga.L[lev];
    const PaBoxDev bx = L.boxes[R.box];
    const PaLayDev ly = L.lay_in[R.box];
    const int a1 = inside ? q % R.n1 : 0, a2 = inside ? q / R.n1 : 0;
    const int d = R.face % 3;
    const int t1 = (d == 0) ? 1 : 0, t2 = (d == 2) ? 1 : 2;
    const int s = (R.face < 3) ? 1 : -1;
    int g[3];
    g[d] = (R.face < 3) ? -1 : bx.n[d];
    g[t1] = a1; g[t2] = a2;
    const long long ga_ = cell_addr(ly, g[0], g[1], g[2]);
    const long long sd = (d == 0) ? 1 : (d == 1) ? (long long)ly.P : (long long)ly.PS;
    if (R.kind != PA_FACE_CF) {                                    // physical walls: nothing to stage (uniform per block)
        if (!active) return;
        for (int m = 0; m < ncomp; ++m) {
            double* p = L.out + ga_ + m * L.cs_in;
            const double v = xform(xf, p[s * sd]);
            *p = (R.kind == PA_FACE_NEUMANN) ? v : -v;
        }
        return;
    }
    // coarse footprint of the chunk [fb.cell0, last] of the face plane, one coarse cell of rim all round
    const int r = R.ratio;
    const int last = (fb.cell0 + PA_FACE_CHUNK < ncell ? fb.cell0 + PA_FACE_CHUNK : ncell) - 1;
    const int row0 = fb.cell0 / R.n1, row1 = last / R.n1;
    const int c0 = (row0 == row1) ? fb.cell0 % R.n1 : 0, c1 = (row0 == row1) ? last % R.n1 : R.n1 - 1;
    const int jc0 = fdiv_dev(bx.lo[t1] + c0, r) - 1, jc1 = fdiv_dev(bx.lo[t1] + c1, r) + 1;
    const int kc0 = fdiv_dev(bx.lo[t2] + row0, r) - 1, kc1 = fdiv_dev(bx.lo[t2] + row1, r) + 1;
    const int W = jc1 - jc0 + 1, Hh = kc1 - kc0 + 1;
    const bool staged = W * Hh <= BCF_TILE;                        // always true for chunks of PA_FACE_CHUNK cells; kept as a guard
    const LevArgs& LC = ga.L[lev - 1];
    const int j = bx.lo[t1] + a1, k = bx.lo[t2] + a2;
    const int jc = fdiv_dev(j, r), kc = fdiv_dev(k, r);
    const long long e0 = R.cidx + (long long)(kc - R.rlo2) * R.rn1 + (jc - R.rlo1);
    const int sc0 = (kc - kc0) * W + (jc - jc0);                   // this cell's coarse cell inside the staged tile
    for (int m = 0; m < ncomp; ++m) {
        const double* cbase = LC.in + m * LC.cs_in;
        if (staged) {
            __syncthreads();                                       // the previous component's readers are done with the tile
            for (int i = threadIdx.x; i < W * Hh; i += PA_FACE_CHUNK) {
                const int jj = jc0 + i % W, kk = kc0 + i / W;
                double v = PA_NAN;                                 // outside the register plane: never read (the flags forbid it)
                if (jj >= R.rlo1 && jj < R.rlo1 + R.rn1 && kk >= R.rlo2 && kk < R.rlo2 + R.rn2)
                    v = crse_val(coff, R.cidx + (long long)(kk - R.rlo2) * R.rn1 + (jj - R.rlo1), cbase, recv, ncomp, m, xf, LC.peers, LC.in_comp + m);
                cs[i] = v;
            }
            __syncthreads();
        }
        if (!active) continue;
        double* p = L.out + ga_ + m * L.cs_in;
#define CR(o1, o2) (staged ? cs[sc0 + (o2) * W + (o1)] : crse_val(coff, e0 + (long long)(o2) * R.rn1 + (o1), cbase, recv, ncomp, m, xf, LC.peers, LC.in_comp + m))
        const double c00 = CR(0, 0);
        int lo = PA_FLAG_NC(fl, 0) ? -1 : 0;
        int hi = PA_FLAG_NC(fl, 1) ? 1 : 0;
        double fac = (hi == lo + 1) ? 1.0 : 0.5;
        const double d1 = fac * (CR(hi, 0) - CR(lo, 0));
        const double d11 = (hi == lo + 2) ? 0.5 * (CR(1, 0) - 2. * c00 + CR(-1, 0)) : 0.;
        lo = PA_FLAG_NC(fl, 2) ? -1 : 0;
        hi = PA_FLAG_NC(fl, 3) ? 1 : 0;
        fac = (hi == lo + 1) ? 1.0 : 0.5;
        const double d2 = fac * (CR(0, hi) - CR(0, lo));
        const double d22 = (hi == lo + 2) ? 0.5 * (CR(0, 1) - 2. * c00 + CR(0, -1)) : 0.;
        const double d12 = (((fl >> 6) & 15u) == 15u)
                               ? 0.25 * (CR(1, 1) - CR(-1, 1) + CR(-1, -1) - CR(1, -1)) : 0.0;
#undef CR
        const double x1 = -0.5 + (j - jc * r + 0.5) / r;
        const double x2 = -0.5 + (k - kc * r + 0.5) / r;
        const double bcval = c00 + x1 * d1 + (x1 * x1) * d11 + x2 * d2 + (x2 * x2) * d22 + x1 * x2 * d12;
        double tmp = 0.0;
        for (int mm = 1; mm < R.nx; ++mm) tmp += xform(xf, p[mm * s * sd]) * R.coef[mm];
        double v = tmp;
        v += bcval * R.coef[0];
        *p = v;
    }
}

cudaError_t launch_bcfill(const PaFaceRec* recs, const int* rec_level, const PaFaceBlock* blocks, long long blk0, long long blk1,
                          const unsigned short* flags, const long long* coff, const GridArgs& ga,
                          int ncomp, const double* recv, GhostXform xf, cudaStream_t st) {
    if (blk1 <= blk0) return cudaSuccess;
    const char* v2 = getenv("PA_BCFILL_V2");
    if (!(v2 && v2[0] == '0'))
        PA_LAUNCH((unsigned)(blk1 - blk0), PA_FACE_CHUNK, 0, st, k_bcfill_v2)(recs, rec_level, blocks + blk0, flags, coff, ga, ncomp, recv, xf);
    else
    PA_LAUNCH((unsigned)(blk1 - blk0), PA_FACE_CHUNK, 0, st, k_bcfill)(recs, rec_level, blocks + blk0, flags, coff, ga, ncomp, recv, xf);
    ++g_launches;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------------
// stencil arithmetic shared by the simple and the TMA kernels (expression order = reference, SURVEY App. B)
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double cdiff(double dxi, double m, double c, double p) {
    // the reference's sequence, sign of zero included: faces f = dxinv*(s(i)-s(i-1)) are multiplied by 1/b = -1
    // (MLCellABecLap::getFluxes), averaged (average_face_to_cellcenter), and multiplied by -1 again (grad.cpp:219).  When the
    // two face differences cancel exactly the result is -0, which 0.5*(fl+fh) would turn into +0.
    const double fl = dxi * (c - m), fh = dxi * (p - c);
    return -(0.5 * ((-fl) + (-fh)));
}

__device__ __forceinline__ double2 ld2(const double* p) { return *reinterpret_cast<const double2*>(p); }
__device__ __forceinline__ void st2(double* p, double a, double b) { *reinterpret_cast<double2*>(p) = make_double2(a, b); }

// Address of input cell (i,j,k) of local box `box` (box-relative; at most one cell outside the valid region, through
// one face).  A ghost cell of a LINKED face is the neighbour's valid cell, read in place (own slab or a peer's);
// otherwise it is this box's materialised ghost cell.  `comp` counts from the first input component.
__device__ __forceinline__ const double* in_ptr(const LevArgs& L, int box, const PaLayDev& li, const PaBoxDev& bx, int comp,
                                                int i, int j, int k) {
    int face = -1;
    if (i < 0) face = 0; else if (i >= bx.n[0]) face = 3;
    else if (j < 0) face = 1; else if (j >= bx.n[1]) face = 4;
    else if (k < 0) face = 2; else if (k >= bx.n[2]) face = 5;
    if (face >= 0) {
        const PaNbrFace F = L.nbr[box].f[face];
        if (F.nb >= 0) {
            const PaPeerSlab ps = L.peers[F.rank];
            return ps.base + (long long)(L.in_comp + comp) * ps.cs + cell_addr(L.lay_in[F.nb], i + F.rel[0], j + F.rel[1], k + F.rel[2]);
        }
    }
    return L.in + (long long)comp * L.cs_in + cell_addr(li, i, j, k);
}

// One tile = rows [y0,y0+ny) x planes [z0,z0+nz) of a box, full x extent.  Each thread handles x pairs with
// 128-bit loads; neighbours come through L1/L2.  This is the general fallback path (any box width) and the
// reference point the TMA pipeline is measured against.
template <int MODE>
__global__ void __launch_bounds__(256) k_stencil_simple(const PaTile* __restrict__ tiles, GridArgs ga, StencilExtra ex) {
    const PaTile t = tiles[blockIdx.x];
    const LevArgs& L = ga.L[t.lev];
    const PaBoxDev bx = L.boxes[t.box];
    const PaLayDev li = L.lay_in[t.box];
    const PaLayDev lo = L.lay_out[t.box];
    const int v = blockIdx.y;
    const int nx = bx.n[0];
    const int nq = (nx + 1) >> 1;
    const int items = nq * t.ny * t.nz;
    const double* __restrict__ in0 = L.in + (MODE == MODE_DIV ? 0 : (long long)v * L.cs_in);
    const int nout = (MODE == MODE_GRAD) ? 4 : (MODE == MODE_DIV ? 1 : 3);
    double* __restrict__ out0 = L.out + (long long)v * nout * L.cs_out;
    const double dxi = L.dxi[0], dyi = L.dxi[1], dzi = L.dxi[2];
    for (int w = threadIdx.x; w < items; w += blockDim.x) {
        const int q = w % nq;
        const int r = w / nq;
        const int jy = t.y0 + r % t.ny, kz = t.z0 + r / t.ny;
        const int i = 2 * q;
        const long long a = cell_addr(li, i, jy, kz);
        const long long o = cell_addr(lo, i, jy, kz);
        const bool two = (i + 1 < nx);
        double r0[4], r1[4];
        const int xe = two ? i + 2 : i + 1;                 // x index of the cell right of this item's last valid cell
        if (MODE != MODE_DIV) {
            const double* p = in0 + a;
            double2 c = ld2(p);
            if (!two) c.y = *in_ptr(L, t.box, li, bx, v, i + 1, jy, kz);
            const double xm = *in_ptr(L, t.box, li, bx, v, i - 1, jy, kz), xp = *in_ptr(L, t.box, li, bx, v, xe, jy, kz);
            const double2 ym = ld2(in_ptr(L, t.box, li, bx, v, i, jy - 1, kz)), yp = ld2(in_ptr(L, t.box, li, bx, v, i, jy + 1, kz));
            const double2 zm = ld2(in_ptr(L, t.box, li, bx, v, i, jy, kz - 1)), zp = ld2(in_ptr(L, t.box, li, bx, v, i, jy, kz + 1));
            const double gx0 = cdiff(dxi, xm, c.x, c.y), gx1 = cdiff(dxi, c.x, c.y, xp);
            const double gy0 = cdiff(dyi, ym.x, c.x, yp.x), gy1 = cdiff(dyi, ym.y, c.y, yp.y);
            const double gz0 = cdiff(dzi, zm.x, c.x, zp.x), gz1 = cdiff(dzi, zm.y, c.y, zp.y);
            if (MODE == MODE_GRAD) {
                r0[0] = gx0; r0[1] = gy0; r0[2] = gz0; r0[3] = sqrt(gx0 * gx0 + gy0 * gy0 + gz0 * gz0);
                r1[0] = gx1; r1[1] = gy1; r1[2] = gz1; r1[3] = sqrt(gx1 * gx1 + gy1 * gy1 + gz1 * gz1);
            } else if (MODE == MODE_GRAD3) {
                r0[0] = gx0; r0[1] = gy0; r0[2] = gz0;
                r1[0] = gx1; r1[1] = gy1; r1[2] = gz1;
            } else {   // MODE_NORMAL
                const double n0 = -fmax(1e-14, sqrt(gx0 * gx0 + gy0 * gy0 + gz0 * gz0));
                const double n1 = -fmax(1e-14, sqrt(gx1 * gx1 + gy1 * gy1 + gz1 * gz1));
                r0[0] = gx0 / n0; r0[1] = gy0 / n0; r0[2] = gz0 / n0;
                r1[0] = gx1 / n1; r1[1] = gy1 / n1; r1[2] = gz1 / n1;
                if (ex.aux[t.lev]) {
                    double* g = ex.aux[t.lev] + o;
                    const long long cg = ex.cs_aux[t.lev];
                    if (two) { st2(g, gx0, gx1); st2(g + cg, gy0, gy1); st2(g + 2 * cg, gz0, gz1); }
                    else { g[0] = gx0; g[cg] = gy0; g[2 * cg] = gz0; }
                }
            }
        } else {
            const double* px = in0 + a;
            const double* py = px + L.cs_in;
            const double* pz = py + L.cs_in;
            double2 cx = ld2(px);
            if (!two) cx.y = *in_ptr(L, t.box, li, bx, 0, i + 1, jy, kz);
            const double xm = *in_ptr(L, t.box, li, bx, 0, i - 1, jy, kz), xp = *in_ptr(L, t.box, li, bx, 0, xe, jy, kz);
            const double2 cy = ld2(py), ym = ld2(in_ptr(L, t.box, li, bx, 1, i, jy - 1, kz)), yp = ld2(in_ptr(L, t.box, li, bx, 1, i, jy + 1, kz));
            const double2 cz = ld2(pz), zm = ld2(in_ptr(L, t.box, li, bx, 2, i, jy, kz - 1)), zp = ld2(in_ptr(L, t.box, li, bx, 2, i, jy, kz + 1));
            const double dx0 = cdiff(dxi, xm, cx.x, cx.y), dx1 = cdiff(dxi, cx.x, cx.y, xp);
            const double dy0 = cdiff(dyi, ym.x, cy.x, yp.x), dy1 = cdiff(dyi, ym.y, cy.y, yp.y);
            const double dz0 = cdiff(dzi, zm.x, cz.x, zp.x), dz1 = cdiff(dzi, zm.y, cz.y, zp.y);
            r0[0] = 0.5 * (((0.0 + dx0) + dy0) + dz0);
            r1[0] = 0.5 * (((0.0 + dx1) + dy1) + dz1);
            if (ex.do_threshold) {
                const double2 pc = ld2(ex.prog[t.lev] + a);
                if (pc.x < ex.threshold || pc.x > 1.0 - ex.threshold) r0[0] = 0.0;
                if (pc.y < ex.threshold || pc.y > 1.0 - ex.threshold) r1[0] = 0.0;
            }
        }
        double* po = out0 + o;
#pragma unroll
        for (int m = 0; m < nout; ++m) {
            if (two) st2(po + m * L.cs_out, r0[m], r1[m]); else po[m * L.cs_out] = r0[m];
        }
    }
}

cudaError_t launch_stencil_simple(int mode, const PaTile* tiles, int ntiles, const GridArgs& ga, const StencilExtra& ex,
                                  int nvar, cudaStream_t st) {
    if (ntiles <= 0) return cudaSuccess;
    dim3 grid(ntiles, nvar), block(256);
    switch (mode) {
        case MODE_GRAD: PA_LAUNCH(grid, block, 0, st, k_stencil_simple<MODE_GRAD>)(tiles, ga, ex); break;
        case MODE_GRAD3: PA_LAUNCH(grid, block, 0, st, k_stencil_simple<MODE_GRAD3>)(tiles, ga, ex); break;
        case MODE_NORMAL: PA_LAUNCH(grid, block, 0, st, k_stencil_simple<MODE_NORMAL>)(tiles, ga, ex); break;
        case MODE_DIV: PA_LAUNCH(grid, block, 0, st, k_stencil_simple<MODE_DIV>)(tiles, ga, ex); break;
        default: return cudaErrorInvalidValue;
    }
    ++g_launches;
    return cudaGetLastError();
}

// K = 0.5 div n on the OUTERMOST cell layer of each box: the cells whose stencil leaves the box, which the fused curvature
// kernel (curv_fused.cu) does not compute.  Arithmetic and ghost rules are MODE_DIV's: a ghost cell of a linked face is the
// neighbour's valid cell read in place, any other one is this box's materialised ghost cell (halo / coarse-fine / wall fill
// of n, curvature.cpp:505-547).  blockIdx.y = entry of the (level, box) list, threads stride over the box's shell cells:
// the two z faces as whole planes, then the y faces of the remaining planes as whole rows, then the x faces cell by cell.
// Boxes are at least 3 cells wide in every direction (the fused path's eligibility rule).
__global__ void __launch_bounds__(256) k_div_shell(const int* __restrict__ box_level, const int* __restrict__ box_index, GridArgs ga, StencilExtra ex) {
    const int lev = box_level[blockIdx.y], box = box_index[blockIdx.y];
    const LevArgs& L = ga.L[lev];
    const PaBoxDev bx = L.boxes[box];
    const PaLayDev li = L.lay_in[box];
    const PaLayDev lo = L.lay_out[box];
    const int nx = bx.n[0], ny = bx.n[1], nz = bx.n[2];
    const long long nA = (long long)nx * ny, nC = (long long)nx * (nz - 2), nE = (long long)(ny - 2) * (nz - 2);
    const long long total = 2 * nA + 2 * nC + 2 * nE;
    const double dxi = L.dxi[0], dyi = L.dxi[1], dzi = L.dxi[2];
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < total; c += (long long)gridDim.x * blockDim.x) {
        int i, j, k;
        long long r = c;
        if (r < 2 * nA) {
            k = (r < nA) ? 0 : nz - 1;
            if (r >= nA) r -= nA;
            i = (int)(r % nx); j = (int)(r / nx);
        } else if ((r -= 2 * nA) < 2 * nC) {
            j = (r < nC) ? 0 : ny - 1;
            if (r >= nC) r -= nC;
            i = (int)(r % nx); k = 1 + (int)(r / nx);
        } else {
            r -= 2 * nC;
            i = (r < nE) ? 0 : nx - 1;
            if (r >= nE) r -= nE;
            j = 1 + (int)(r % (ny - 2)); k = 1 + (int)(r / (ny - 2));
        }
        const double cx = *in_ptr(L, box, li, bx, 0, i, j, k), xm = *in_ptr(L, box, li, bx, 0, i - 1, j, k), xp = *in_ptr(L, box, li, bx, 0, i + 1, j, k);
        const double cy = *in_ptr(L, box, li, bx, 1, i, j, k), ym = *in_ptr(L, box, li, bx, 1, i, j - 1, k), yp = *in_ptr(L, box, li, bx, 1, i, j + 1, k);
        const double cz = *in_ptr(L, box, li, bx, 2, i, j, k), zm = *in_ptr(L, box, li, bx, 2, i, j, k - 1), zp = *in_ptr(L, box, li, bx, 2, i, j, k + 1);
        const double dx = cdiff(dxi, xm, cx, xp), dy = cdiff(dyi, ym, cy, yp), dz = cdiff(dzi, zm, cz, zp);
        double kk = 0.5 * (((0.0 + dx) + dy) + dz);
        if (ex.do_threshold) {
            const double pc = ex.prog[lev][cell_addr(li, i, j, k)];
            if (pc < ex.threshold || pc > 1.0 - ex.threshold) kk = 0.0;
        }
        L.out[cell_addr(lo, i, j, k)] = kk;
    }
}
cudaError_t launch_div_shell(const int* box_level, const int* box_index, int nboxes, int blocks_per_box, const GridArgs& ga,
                             const StencilExtra& ex, cudaStream_t st) {
    if (nboxes <= 0) return cudaSuccess;
    PA_LAUNCH(dim3(blocks_per_box, nboxes), 256, 0, st, k_div_shell)(box_level, box_index, ga, ex);
    ++g_launches;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------------
// pointwise passes of the curvature tool
// ------------------------------------------------------------------------------------------------------------
// one thread per x pair of a valid row; boxes enumerated through blockIdx.y
template <class F>
__device__ __forceinline__ void for_valid_cells(const PaBoxDev& b, F&& f) {
    const long long n = (long long)b.n[0] * b.n[1] * b.n[2];
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
        int i = (int)(c % b.n[0]);
        long long r = c / b.n[0];
        f(i, (int)(r % b.n[1]), (int)(r / b.n[1]));
    }
}

// Order-independent 64-bit fingerprint of the VALID cells of a level: sum (mod 2^64) over components, boxes and cells of
// mix(bit pattern ^ mix(level, GLOBAL box id, component, cell)).  Each rank sums its own boxes; the wrapped sum of the
// ranks' values is the same for any box -> rank map exactly when every output bit is the same (bench.py: output_hash).
__device__ __forceinline__ unsigned long long hmix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ULL; z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL; z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__global__ void __launch_bounds__(256) k_field_hash(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay, const int* __restrict__ gid,
                                                    const double* __restrict__ base, long long cs, int comp0, int ncomp, int lev,
                                                    unsigned long long* __restrict__ out) {
    const PaBoxDev b = boxes[blockIdx.y];
    const PaLayDev y = lay[blockIdx.y];
    const unsigned long long g = (unsigned long long)gid[blockIdx.y];
    unsigned long long acc = 0;
    for (int m = 0; m < ncomp; ++m) {
        const unsigned long long key = hmix64(((unsigned long long)lev << 56) ^ (g << 16) ^ (unsigned long long)(comp0 + m));
        const double* p = base + (long long)m * cs;
        for_valid_cells(b, [&](int i, int j, int k) {
            const unsigned long long cell = ((unsigned long long)k * b.n[1] + j) * b.n[0] + i;
            acc += hmix64((unsigned long long)__double_as_longlong(p[cell_addr(y, i, j, k)]) ^ hmix64(key + cell));
        });
    }
    // block sum, then one atomic per block
    __shared__ unsigned long long part[256];
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) part[threadIdx.x] += part[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) atomicAdd(out, part[0]);
}
cudaError_t launch_field_hash(const PaBoxDev* boxes, const PaLayDev* lay, const int* gid, int nboxes, const double* base, long long cs,
                              int comp0, int ncomp, int lev, unsigned long long* out, cudaStream_t st) {
    for (int b0 = 0; b0 < nboxes; b0 += 65535) {
        const int n = nboxes - b0 < 65535 ? nboxes - b0 : 65535;
        PA_LAUNCH(dim3(96, n), 256, 0, st, k_field_hash)(boxes + b0, lay + b0, gid + b0, base, cs, comp0, ncomp, lev, out);
        ++g_launches;
    }
    return cudaGetLastError();
}

// Progress variable c = (S - progMin) * invdenom on valid cells (curvature.cpp:310-321)
__global__ void k_progress(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay_in,
                           const PaLayDev* __restrict__ lay_out, const double* __restrict__ S, double* __restrict__ C,
                           double pmin, double invdenom) {
    const PaBoxDev b = boxes[blockIdx.y];
    const PaLayDev yi = lay_in[blockIdx.y], yo = lay_out[blockIdx.y];
    for_valid_cells(b, [&](int i, int j, int k) { C[cell_addr(yo, i, j, k)] = (S[cell_addr(yi, i, j, k)] - pmin) * invdenom; });
}
cudaError_t launch_progress(const PaBoxDev* boxes, const PaLayDev* lay_in, const PaLayDev* lay_out, int nboxes,
                            const double* S, double* C, double pmin, double invdenom, cudaStream_t st) {
    if (nboxes <= 0) return cudaSuccess;
    PA_LAUNCH(dim3(32, nboxes), 256, 0, st, k_progress)(boxes, lay_in, lay_out, S, C, pmin, invdenom);
    ++g_launches;
    return cudaGetLastError();
}

// threshold clip of the flame normal, in place, after K of the level is done (curvature.cpp:549-567)
__global__ void k_clip_normal(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay_c,
                              const PaLayDev* __restrict__ lay_n, const double* __restrict__ C, double* __restrict__ N,
                              long long cs_n, double thr) {
    const PaBoxDev b = boxes[blockIdx.y];
    const PaLayDev yc = lay_c[blockIdx.y], yn = lay_n[blockIdx.y];
    for_valid_cells(b, [&](int i, int j, int k) {
        const double c = C[cell_addr(yc, i, j, k)];
        if (c < thr || c > 1.0 - thr) {
            const long long a = cell_addr(yn, i, j, k);
            N[a] = 0.0; N[a + cs_n] = 0.0; N[a + 2 * cs_n] = 0.0;
        }
    });
}
cudaError_t launch_clip_normal(const PaBoxDev* boxes, const PaLayDev* lay_c, const PaLayDev* lay_n, int nboxes,
                               const double* C, double* N, long long cs_n, double thr, cudaStream_t st) {
    if (nboxes <= 0) return cudaSuccess;
    PA_LAUNCH(dim3(32, nboxes), 256, 0, st, k_clip_normal)(boxes, lay_c, lay_n, C, N, cs_n, thr);
    ++g_launches;
    return cudaGetLastError();
}

// Gaussian curvature n.adj(H).n / |grad c|^4 (curvature.cpp:615-672).  G = un-normalised gradient (3 comps),
// H = Hessian rows (9 comps: d(G_i)/dx_j at comp 3i+j).  nrm is recomputed exactly as pass 1 did.
__global__ void k_gauss(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay, const PaLayDev* __restrict__ lay_c,
                        const double* __restrict__ G, long long cg, const double* __restrict__ H, long long ch,
                        const double* __restrict__ C, double* __restrict__ Kg, int do_thr, double thr) {
    const PaBoxDev b = boxes[blockIdx.y];
    const PaLayDev y = lay[blockIdx.y], yc = lay_c[blockIdx.y];
    for_valid_cells(b, [&](int i, int j, int k) {
        const long long a = cell_addr(y, i, j, k);
        const double Cx = G[a], Cy = G[a + cg], Cz = G[a + 2 * cg];
        const double Hx0 = H[a], Hx1 = H[a + ch], Hx2 = H[a + 2 * ch];
        const double Hy0 = H[a + 3 * ch], Hy1 = H[a + 4 * ch], Hy2 = H[a + 5 * ch];
        const double Hz0 = H[a + 6 * ch], Hz1 = H[a + 7 * ch], Hz2 = H[a + 8 * ch];
        const double Ax0 = Hy1 * Hz2 - Hz1 * Hy2;
        const double Ay0 = Hy2 * Hz0 - Hz2 * Hy0;
        const double Az0 = Hy0 * Hz1 - Hz0 * Hy1;
        const double Ax1 = Hx2 * Hz1 - Hz2 * Hx1;
        const double Ay1 = Hx0 * Hz2 - Hz0 * Hx2;
        const double Az1 = Hx1 * Hz0 - Hz1 * Hx0;
        const double Ax2 = Hx1 * Hy2 - Hy1 * Hx2;
        const double Ay2 = Hx2 * Hy0 - Hy2 * Hx0;
        const double Az2 = Hx0 * Hy1 - Hy0 * Hx1;
        const double nrm = -fmax(1e-14, sqrt(Cx * Cx + Cy * Cy + Cz * Cz));
        double v = (Cx * (Ax0 * Cx + Ax1 * Cy + Ax2 * Cz) + Cy * (Ay0 * Cx + Ay1 * Cy + Ay2 * Cz) +
                    Cz * (Az0 * Cx + Az1 * Cy + Az2 * Cz)) / pow(nrm, 4.0);
        if (do_thr) {
            const double c = C[cell_addr(yc, i, j, k)];
            if (c < thr || c > 1.0 - thr) v = 0.0;
        }
        Kg[a] = v;
    });
}
cudaError_t launch_gauss(const PaBoxDev* boxes, const PaLayDev* lay, const PaLayDev* lay_c, int nboxes, const double* G,
                         long long cs_g, const double* H, long long cs_h, const double* C, double* Kg, int do_thr,
                         double thr, cudaStream_t st) {
    if (nboxes <= 0) return cudaSuccess;
    PA_LAUNCH(dim3(32, nboxes), 256, 0, st, k_gauss)(boxes, lay, lay_c, G, cs_g, H, cs_h, C, Kg, do_thr, thr);
    ++g_launches;
    return cudaGetLastError();
}

// StrainRate as the reference actually computes it: the -nn:grad(u) term is overwritten, leaving div u
// (curvature.cpp:736-747).
__global__ void k_strain(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay, const double* __restrict__ dU,
                         long long cs, double* __restrict__ sr) {
    const PaBoxDev b = boxes[blockIdx.y];
    const PaLayDev y = lay[blockIdx.y];
    for_valid_cells(b, [&](int i, int j, int k) {
        const long long a = cell_addr(y, i, j, k);
        sr[a] = dU[a] + dU[a + 4 * cs] + dU[a + 8 * cs];
    });
}
cudaError_t launch_strain(const PaBoxDev* boxes, const PaLayDev* lay, int nboxes, const double* dU, long long cs,
                          double* sr, cudaStream_t st) {
    if (nboxes <= 0) return cudaSuccess;
    PA_LAUNCH(dim3(32, nboxes), 256, 0, st, k_strain)(boxes, lay, dU, cs, sr);
    ++g_launches;
    return cudaGetLastError();
}

// VelFlameNormal = u.n with the (already clipped) normal (curvature.cpp:761-789)
__global__ void k_velnormal(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay_u, const PaLayDev* __restrict__ lay_n,
                            const PaLayDev* __restrict__ lay_o, const double* __restrict__ U, long long cu,
                            const double* __restrict__ N, long long cn, const double* __restrict__ C,
                            double* __restrict__ out, int do_thr, double thr) {
    const PaBoxDev b = boxes[blockIdx.y];
    const PaLayDev yu = lay_u[blockIdx.y], yn = lay_n[blockIdx.y], yo = lay_o[blockIdx.y];
    for_valid_cells(b, [&](int i, int j, int k) {
        const long long au = cell_addr(yu, i, j, k), an = cell_addr(yn, i, j, k);
        double v = U[au] * N[an] + U[au + cu] * N[an + cn] + U[au + 2 * cu] * N[an + 2 * cn];
        if (do_thr) {
            const double c = C[an];
            if (c < thr || c > 1.0 - thr) v = 0.0;
        }
        out[cell_addr(yo, i, j, k)] = v;
    });
}
cudaError_t launch_velnormal(const PaBoxDev* boxes, const PaLayDev* lay_u, const PaLayDev* lay_n, const PaLayDev* lay_o,
                             int nboxes, const double* U, long long cs_u, const double* N, long long cs_n,
                             const double* C, double* out, int do_thr, double thr, cudaStream_t st) {
    if (nboxes <= 0) return cudaSuccess;
    PA_LAUNCH(dim3(32, nboxes), 256, 0, st, k_velnormal)(boxes, lay_u, lay_n, lay_o, U, cs_u, N, cs_n, C, out, do_thr, thr);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace pa

// The kernels of the composite implicit-diffusion solve (pa_smooth) live in smooth.cu and are compiled in this translation
// unit: they use the layout addressing above, and the library is built from a fixed list of translation units.
#include "smooth.cu"
