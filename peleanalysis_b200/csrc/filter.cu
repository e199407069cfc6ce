// filter.cu -- device side of the filterPlt path (R/Src/filterPlt.cpp:166-221): ghost cells of a level by FillPatch rules,
// then PelePhysics' Filter on every box.  R = /root/reference, AX = its vendored amrex/Src, PP = PelePhysics/Source.
//
//   k_fp_gather   coarse VALID cells -> coarse patches of the pieces (FillPatchSingleLevel into mf_crse_patch,
//                 AX/AmrCore/AMReX_FillPatchUtil_I.H), one thread per coarse cell over the copy-tag table
//   k_fp_unpack   several ranks: cells of other ranks' boxes (packed by the exchange pack kernel, moved by the caller) ->
//                 ghost cells of local boxes and coarse patches (FillPatchTwoLevels' ParallelCopy / FillBoundary data)
//   k_fp_interp   pieces <- coarse patches: MFCellConsLinInterp with the monotonised-central slope
//                 (AX/AmrCore/AMReX_MFInterp_3D_C.H:178-260) or MFPCInterp; coarse reads clamp their index into the coarse
//                 domain, which IS the first-order extrapolation the reference applies to the patch (AMReX_FilCC_3D_C.H)
//   k_fp_clamp    ghost cells outside the domain <- the cell at the clamped index of the same FAB (faces, edges, corners:
//                 AX/Base/AMReX_PhysBCFunct.H:406-640 ends in exactly that)
//   k_filter      qh = 0; for n, m, l: qh += ((w[l] * w[m]) * w[n]) * q(i+l, j+m, k+n)   (PP/Utility/Filter/Filter.H:28-50)
//
// All arithmetic keeps the reference's operation order with separate IEEE multiplies and adds (-fmad=false): results are
// bit-identical to the reference's CPU build.  The same-level copies of the fill are the library's FillBoundary table
// (k_halo, all ghost layers).  These are gather kernels over precomputed descriptor tables (hier.cpp: Hier::fill_patch);
// the filter is a dense (2g+1)^3 weighted sum whose bound is the FP64 pipe for g >= 2 and HBM for g = 1.
#include <algorithm>
#include <cstdint>

#include "kernels.cuh"

namespace pa {

namespace {

__device__ __forceinline__ long long lay_addr(const PaLayDev& y, int i, int j, int k) {
    return y.off + (long long)(k + y.ng) * y.PS + (long long)(j + y.ng) * y.P + (i + y.ng + y.xoff);
}
// last index in [0, n) whose start is <= c
template <class T, class F>
__device__ __forceinline__ int last_le(const T* a, int n, long long c, F start) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (start(a[mid]) <= c) lo = mid; else hi = mid - 1;
    }
    return lo;
}
static inline int blocks_for(long long n, int block, int cap = 148 * 16) {
    long long g = (n + block - 1) / block;
    return (int)std::max<long long>(1, std::min<long long>(g, cap));
}
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
#ifdef PA_HOST_EMULATION
__device__ __forceinline__ double ldro(const double* p) { return *p; }
#else
__device__ __forceinline__ double ldro(const double* p) { return __ldg(p); }      // read-only path, L1-cached
#endif

__global__ void k_fp_gather(const PaFpCopy* __restrict__ copies, int ncopies, long long ncells, const PaFpPiece* __restrict__ pieces,
                            const PaBoxDev* __restrict__ cboxes, const PaLayDev* __restrict__ clay, const double* __restrict__ cbase,
                            long long ccs, int ncomp, double* __restrict__ scratch, long long ncrse) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        const PaFpCopy t = copies[last_le(copies, ncopies, c, [](const PaFpCopy& x) { return x.start; })];
        const long long q = c - t.start;
        const int i = (int)(q % t.n[0]);
        const long long r = q / t.n[0];
        const int j = (int)(r % t.n[1]), k = (int)(r / t.n[1]);
        const int ci = t.lo[0] + i, cj = t.lo[1] + j, ck = t.lo[2] + k;
        const PaFpPiece P = pieces[t.piece];
        const long long dst = P.cstart + ((long long)(ck - P.clo[2]) * P.cn[1] + (cj - P.clo[1])) * P.cn[0] + (ci - P.clo[0]);
        const PaBoxDev sb = cboxes[t.sbox];
        const long long sa = lay_addr(clay[t.sbox], ci - sb.lo[0], cj - sb.lo[1], ck - sb.lo[2]);
        for (int m = 0; m < ncomp; ++m) scratch[dst + m * ncrse] = cbase[sa + m * ccs];
    }
}

// Several ranks: the fill's sources owned by another rank arrive packed in the recv slab ([cell][comp], the exchange pack
// kernel's layout).  One thread per slab cell over the unpack table: into a ghost cell of a local box (same-level source) or a
// coarse-patch cell of a piece (coarse source).  Runs before the interpolation, which reads the coarse patches.
__global__ void k_fp_unpack(const PaFpUnpack* __restrict__ recs, int nrecs, long long ncells, const double* __restrict__ recv,
                            const PaFpPiece* __restrict__ pieces, double* __restrict__ scratch, long long ncrse,
                            const PaBoxDev* __restrict__ fboxes, const PaLayDev* __restrict__ flay, double* __restrict__ fbase,
                            long long fcs, int ncomp) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        const PaFpUnpack t = recs[last_le(recs, nrecs, c, [](const PaFpUnpack& x) { return x.start; })];
        const long long q = c - t.start;
        const int i = t.lo[0] + (int)(q % t.n[0]);
        const long long r = q / t.n[0];
        const int j = t.lo[1] + (int)(r % t.n[1]), k = t.lo[2] + (int)(r / t.n[1]);
        const double* s = recv + (t.rsrc + q) * ncomp;
        if (t.box >= 0) {
            const PaBoxDev b = fboxes[t.box];
            const long long da = lay_addr(flay[t.box], i - b.lo[0], j - b.lo[1], k - b.lo[2]);
            for (int m = 0; m < ncomp; ++m) fbase[da + m * fcs] = s[m];
        } else {
            const PaFpPiece P = pieces[-1 - t.box];
            const long long dst = P.cstart + ((long long)(k - P.clo[2]) * P.cn[1] + (j - P.clo[1])) * P.cn[0] + (i - P.clo[0]);
            for (int m = 0; m < ncomp; ++m) scratch[dst + m * ncrse] = s[m];
        }
    }
}

// Same-level copies of the fill, one thread block per (tag, slice): the tag and the two boxes' records are read once per block
// instead of being searched for and reloaded by every cell's thread (k_halo's general form costs a 14-step binary search over
// ~13 k tags per ghost cell on 512 boxes with 4 ghost layers: 0.31 ms for 16 M cells).  Local sources only, no value transform:
// what the filterPlt path needs.  Cells of a tag are walked row by row (x fastest), so loads and stores of a row are contiguous.
__global__ void __launch_bounds__(128) k_halo_blk(const PaHaloTag* __restrict__ tags, const PaBoxDev* __restrict__ boxes,
                                                  const PaLayDev* __restrict__ lay, double* __restrict__ base, long long cs, int ncomp) {
    const PaHaloTag t = tags[blockIdx.x];
    if (t.sbox < 0) return;                                           // never on a single-rank hierarchy
    const PaBoxDev db = boxes[t.dbox], sb = boxes[t.sbox];
    const PaLayDev dl = lay[t.dbox], sl = lay[t.sbox];
    const int nrows = t.n[1] * t.n[2];
    const long long d0 = lay_addr(dl, t.dlo[0] - db.lo[0], t.dlo[1] - db.lo[1], t.dlo[2] - db.lo[2]);
    const long long s0 = lay_addr(sl, t.dlo[0] + t.shift[0] - sb.lo[0], t.dlo[1] + t.shift[1] - sb.lo[1], t.dlo[2] + t.shift[2] - sb.lo[2]);
    if (t.n[0] >= 16) {                                               // long rows: a warp per row, lanes along x
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
        for (int r = blockIdx.y * nw + warp; r < nrows; r += gridDim.y * nw) {
            const int j = r % t.n[1], k = r / t.n[1];
            const long long da = d0 + (long long)k * dl.PS + (long long)j * dl.P, sa = s0 + (long long)k * sl.PS + (long long)j * sl.P;
            for (int m = 0; m < ncomp; ++m)
                for (int i = lane; i < t.n[0]; i += 32) base[da + i + m * cs] = base[sa + i + m * cs];
        }
    } else {                                                          // thin tags (x faces, edges, corners): a thread per cell
        const int ncell = nrows * t.n[0];
        for (int c = blockIdx.y * blockDim.x + threadIdx.x; c < ncell; c += gridDim.y * blockDim.x) {
            const int i = c % t.n[0], r = c / t.n[0];
            const int j = r % t.n[1], k = r / t.n[1];
            const long long da = d0 + (long long)k * dl.PS + (long long)j * dl.P + i, sa = s0 + (long long)k * sl.PS + (long long)j * sl.P + i;
            for (int m = 0; m < ncomp; ++m) base[da + m * cs] = base[sa + m * cs];
        }
    }
}

struct Dom { int lo[3], hi[3]; };

// the reference's monotonised-central slope of one direction (AMReX_MFInterp_3D_C.H:190-196); amrex::min is std::min
__device__ __forceinline__ double mc_slope(double um, double u0, double up) {
    const double dc = 0.5 * (up - um);
    const double df = 2.0 * (up - u0);
    const double db = 2.0 * (u0 - um);
    const double adf = fabs(df), adb = fabs(db), adc = fabs(dc);
    double s = (df * db >= 0.0) ? (adb < adf ? adb : adf) : 0.0;
    return copysign(1.0, dc) * (adc < s ? adc : s);
}

template <bool CONS>
__global__ void k_fp_interp(const PaFpPiece* __restrict__ pieces, int npieces, long long ncells, const double* __restrict__ scratch,
                            long long ncrse, Dom cdom, int ratio, const PaBoxDev* __restrict__ fboxes, const PaLayDev* __restrict__ flay,
                            double* __restrict__ fbase, long long fcs, int ncomp) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        const PaFpPiece P = pieces[last_le(pieces, npieces, c, [](const PaFpPiece& x) { return x.fstart; })];
        const long long q = c - P.fstart;
        const int i = P.lo[0] + (int)(q % P.n[0]);
        const long long rr = q / P.n[0];
        const int j = P.lo[1] + (int)(rr % P.n[1]), k = P.lo[2] + (int)(rr / P.n[1]);
        const int ic = (i < 0) ? -((-i + ratio - 1) / ratio) : i / ratio;
        const int jc = (j < 0) ? -((-j + ratio - 1) / ratio) : j / ratio;
        const int kc = (k < 0) ? -((-k + ratio - 1) / ratio) : k / ratio;
        const PaBoxDev fb = fboxes[P.box];
        const long long da = lay_addr(flay[P.box], i - fb.lo[0], j - fb.lo[1], k - fb.lo[2]);
        // coarse patch element, index clamped into the coarse domain (first-order extrapolation of the patch)
        auto U = [&](int a, int b, int d) -> long long {
            a = clampi(a, cdom.lo[0], cdom.hi[0]); b = clampi(b, cdom.lo[1], cdom.hi[1]); d = clampi(d, cdom.lo[2], cdom.hi[2]);
            return P.cstart + ((long long)(d - P.clo[2]) * P.cn[1] + (b - P.clo[1])) * P.cn[0] + (a - P.clo[0]);
        };
        for (int m = 0; m < ncomp; ++m) {
            const double* u = scratch + m * ncrse;
            const double u0 = u[U(ic, jc, kc)];
            if (!CONS) { fbase[da + m * fcs] = u0; continue; }                       // MFPCInterp
            const double sx = mc_slope(u[U(ic - 1, jc, kc)], u0, u[U(ic + 1, jc, kc)]);
            const double sy = mc_slope(u[U(ic, jc - 1, kc)], u0, u[U(ic, jc + 1, kc)]);
            const double sz = mc_slope(u[U(ic, jc, kc - 1)], u0, u[U(ic, jc, kc + 1)]);
            double alpha = 1.0;
            if (sx != 0.0 || sy != 0.0 || sz != 0.0) {                               // :216-238
                const double rm1 = (double)(ratio - 1), r2 = (double)(2 * ratio);
                const double dumax = (fabs(sx) * rm1) / r2 + (fabs(sy) * rm1) / r2 + (fabs(sz) * rm1) / r2;
                double umax = u0, umin = u0;
                for (int kk = -1; kk <= 1; ++kk)
                    for (int jj = -1; jj <= 1; ++jj)
                        for (int ii = -1; ii <= 1; ++ii) {
                            const double v = u[U(ic + ii, jc + jj, kc + kk)];
                            umin = (v < umin) ? v : umin;
                            umax = (umax < v) ? v : umax;
                        }
                if (dumax * alpha > (umax - u0)) alpha = (umax - u0) / dumax;
                if (dumax * alpha > (u0 - umin)) alpha = (u0 - umin) / dumax;
            }
            const double slx = sx * alpha, sly = sy * alpha, slz = sz * alpha;
            const double xoff = ((double)(i - ic * ratio) + 0.5) / (double)ratio - 0.5;      // :253-259
            const double yoff = ((double)(j - jc * ratio) + 0.5) / (double)ratio - 0.5;
            const double zoff = ((double)(k - kc * ratio) + 0.5) / (double)ratio - 0.5;
            fbase[da + m * fcs] = ((u0 + xoff * slx) + yoff * sly) + zoff * slz;
        }
    }
}

__global__ void k_fp_clamp(const PaFpClamp* __restrict__ clamps, int nclamps, long long ncells, Dom dom, int g,
                           const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay, double* __restrict__ base,
                           long long cs, int ncomp) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        const PaFpClamp t = clamps[last_le(clamps, nclamps, c, [](const PaFpClamp& x) { return x.start; })];
        const PaBoxDev b = boxes[t.box];
        const int gx = b.n[0] + 2 * g, gy = b.n[1] + 2 * g;
        const long long q = c - t.start;
        const int i = b.lo[0] - g + (int)(q % gx);
        const long long r = q / gx;
        const int j = b.lo[1] - g + (int)(r % gy), k = b.lo[2] - g + (int)(r / gy);
        const int ci = clampi(i, dom.lo[0], dom.hi[0]), cj = clampi(j, dom.lo[1], dom.hi[1]), ck = clampi(k, dom.lo[2], dom.hi[2]);
        if (ci == i && cj == j && ck == k) continue;                                  // inside the domain
        const long long da = lay_addr(lay[t.box], i - b.lo[0], j - b.lo[1], k - b.lo[2]);
        const long long sa = lay_addr(lay[t.box], ci - b.lo[0], cj - b.lo[1], ck - b.lo[2]);
        for (int m = 0; m < ncomp; ++m) base[da + m * cs] = base[sa + m * cs];
    }
}

// ---- the filter -------------------------------------------------------------------------------------------------------
// One thread = a block of four consecutive x cells by two consecutive rows of one (box, component, k): eight independent
// accumulation chains.  For every z offset n the thread walks the 2g + 2 input rows the block touches; a row's 4 + 2g values
// arrive as aligned 128-bit loads and feed BOTH output rows (as y offset m for the upper one and m - 1 for the lower one), and a
// weight row w3[n][m][*] is fetched from shared memory once and serves two consecutive input rows the same way.  Every chain
// still sees its terms in the reference's order (n, then m, then l ascending).  The weight products ((w[l] * w[m]) * w[n]) are
// formed once on the host in that order -- they are the leading factors of the reference's left-to-right product.
// Measured on a B200 (profiles/r02_filter_*): the first version (one row per thread, 64-bit loads at a 32-byte lane stride) was
// bound by L1 throughput at a third of the FP64 pipe; see DESIGN.md section 9.
// G > 0: ghost width known at compile time; G == 0 and ragged blocks (nx not a multiple of 4, odd last row): plain loops.
constexpr int FILTER_THREADS = 128;
constexpr int FILTER_MAX_W3 = 17 * 17 * 17;           // ghost width <= 8 in shared memory; wider filters read w3 from global memory

template <int G>
__global__ void __launch_bounds__(FILTER_THREADS) k_filter(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lin,
                                                            const PaLayDev* __restrict__ lout, int nboxes,
                                                            const long long* __restrict__ work_prefix /* nboxes+1: blocks of 4 x 2 cells */,
                                                            const double* __restrict__ in, long long cs_in, double* __restrict__ out,
                                                            long long cs_out, int ncomp, const double* __restrict__ w3g, int g_rt) {
    const int g = G > 0 ? G : g_rt;
    const int W = 2 * g + 1;
    PA_DYN_SMEM(smem_raw);
    double* w3s = reinterpret_cast<double*>(smem_raw);
    const bool w_in_smem = W * W * W <= FILTER_MAX_W3;
    if (w_in_smem) {
        for (int t = threadIdx.x; t < W * W * W; t += blockDim.x) w3s[t] = w3g[t];
        __syncthreads();
    }
    const double* __restrict__ w3 = w_in_smem ? w3s : w3g;
    const long long per_comp = work_prefix[nboxes];
    const long long nwork = per_comp * ncomp;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < nwork; c += (long long)gridDim.x * blockDim.x) {
        const int m = (int)(c / per_comp);                            // component-major: a component's boxes are contiguous work
        const long long cw = c - (long long)m * per_comp;
        int lo = 0, hi = nboxes - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (work_prefix[mid] <= cw) lo = mid; else hi = mid - 1; }
        const PaBoxDev b = boxes[lo];
        const int nq = (b.n[0] + 3) >> 2, nr = (b.n[1] + 1) >> 1;
        const long long q = cw - work_prefix[lo];
        const int xq = (int)(q % nq);
        const long long r = q / nq;
        const int j = 2 * (int)(r % nr), k = (int)(r / nr);
        const int x0 = 4 * xq;
        const int nv = b.n[0] - x0 >= 4 ? 4 : b.n[0] - x0;
        const int nrow = b.n[1] - j >= 2 ? 2 : 1;
        const PaLayDev yi = lin[lo];
        const double* __restrict__ src = in + (long long)m * cs_in + lay_addr(yi, x0 - g, j - g, k - g);
        double* dst = out + (long long)m * cs_out + lay_addr(lout[lo], x0, j, k);
        const int Pout = lout[lo].P;
        if (G > 0 && nv == 4 && nrow == 2) {
            constexpr int GG = G > 0 ? G : 1;
            constexpr int A = GG & 1;                                 // one leading element more keeps the row segment 16-byte aligned
            constexpr int NV = 4 + 2 * GG + 2 * A;
            constexpr int WW = 2 * GG + 1;
            double a0[4] = {0.0, 0.0, 0.0, 0.0}, a1[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 1
            for (int n = 0; n < WW; ++n) {
                const double* __restrict__ plane = src + (long long)n * yi.PS - A;
                const double* __restrict__ wn = w3 + n * WW * WW;
                double wprev[WW];
#pragma unroll
                for (int l = 0; l < WW; ++l) wprev[l] = 0.0;
#pragma unroll 2
                for (int rr = 0; rr < WW + 1; ++rr) {                 // input row j - g + rr
                    double v[NV];
                    const double2* __restrict__ row2 = reinterpret_cast<const double2*>(plane + (long long)rr * yi.P);
#pragma unroll
                    for (int t = 0; t < NV / 2; ++t) {
#ifdef PA_HOST_EMULATION
                        const double2 p2 = row2[t];
#else
                        const double2 p2 = __ldg(row2 + t);
#endif
                        v[2 * t] = p2.x; v[2 * t + 1] = p2.y;
                    }
                    double wcur[WW];
                    if (rr < WW) {
#pragma unroll
                        for (int l = 0; l < WW; ++l) wcur[l] = wn[rr * WW + l];
#pragma unroll
                        for (int l = 0; l < WW; ++l) {
#pragma unroll
                            for (int t = 0; t < 4; ++t) a0[t] = a0[t] + wcur[l] * v[A + t + l];
                        }
                    }
                    if (rr > 0) {
#pragma unroll
                        for (int l = 0; l < WW; ++l) {
#pragma unroll
                            for (int t = 0; t < 4; ++t) a1[t] = a1[t] + wprev[l] * v[A + t + l];
                        }
                    }
#pragma unroll
                    for (int l = 0; l < WW; ++l) wprev[l] = wcur[l];
                }
            }
            *reinterpret_cast<double2*>(dst) = make_double2(a0[0], a0[1]);
            *reinterpret_cast<double2*>(dst + 2) = make_double2(a0[2], a0[3]);
            *reinterpret_cast<double2*>(dst + Pout) = make_double2(a1[0], a1[1]);
            *reinterpret_cast<double2*>(dst + Pout + 2) = make_double2(a1[2], a1[3]);
        } else {
            for (int rw = 0; rw < nrow; ++rw) {
                double acc[4] = {0.0, 0.0, 0.0, 0.0};
                for (int n = 0; n < W; ++n)
                    for (int mm = 0; mm < W; ++mm) {
                        const double* __restrict__ row = src + (long long)n * yi.PS + (long long)(mm + rw) * yi.P;
                        const double* __restrict__ wr = w3 + (n * W + mm) * W;
                        for (int l = 0; l < W; ++l) {
                            const double w = wr[l];
                            for (int t = 0; t < nv; ++t) acc[t] = acc[t] + w * ldro(row + t + l);
                        }
                    }
                for (int t = 0; t < nv; ++t) dst[(long long)rw * Pout + t] = acc[t];
            }
        }
    }
}

// FP64 pipe rate with the filter's instruction mix (separate multiplies and adds, no FMA): 8 independent chains per thread.
// The measured roofline denominator of k_filter for ghost widths >= 2 (bench.py); results are written so nothing is optimised away.
__global__ void k_fp64_rate(double* __restrict__ out, int iters, double seed) {
    double a[8], w = 1.0 + seed * 1e-9;
#pragma unroll
    for (int t = 0; t < 8; ++t) a[t] = seed + t + threadIdx.x;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int t = 0; t < 8; ++t) a[t] = a[t] + w * a[(t + 1) & 7];
    }
    double s = 0.0;
#pragma unroll
    for (int t = 0; t < 8; ++t) s += a[t];
    out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace

cudaError_t launch_fp64_rate(double* out, int blocks, int threads, int iters, cudaStream_t st) {
    PA_LAUNCH(blocks, threads, 0, st, k_fp64_rate)(out, iters, 0.5);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_halo_blocks(const PaHaloTag* tags, int ntags, int slices, const PaBoxDev* boxes, const PaLayDev* lay, double* base,
                               long long cs, int ncomp, cudaStream_t st) {
    if (ntags <= 0) return cudaSuccess;
    for (int t0 = 0; t0 < ntags; t0 += 65535 * 32) {                   // grid.x limit is 2^31-1; keep launches modest anyway
        const int n = std::min(ntags - t0, 65535 * 32);
        dim3 grid((unsigned)n, (unsigned)std::max(1, std::min(slices, 64)));
        PA_LAUNCH(grid, 128, 0, st, k_halo_blk)(tags + t0, boxes, lay, base, cs, ncomp);
        ++g_launches;
    }
    return cudaGetLastError();
}

cudaError_t launch_fp_gather(const PaFpCopy* copies, int ncopies, long long ncells, const PaFpPiece* pieces, const PaBoxDev* cboxes,
                             const PaLayDev* clay, const double* cbase, long long ccs, int ncomp, double* scratch, long long ncrse,
                             cudaStream_t st) {
    if (ncells <= 0 || ncopies <= 0) return cudaSuccess;
    PA_LAUNCH(blocks_for(ncells, 256), 256, 0, st, k_fp_gather)(copies, ncopies, ncells, pieces, cboxes, clay, cbase, ccs, ncomp, scratch, ncrse);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_fp_unpack(const PaFpUnpack* recs, int nrecs, long long ncells, const double* recv, const PaFpPiece* pieces,
                             double* scratch, long long ncrse, const PaBoxDev* fboxes, const PaLayDev* flay, double* fbase, long long fcs,
                             int ncomp, cudaStream_t st) {
    if (ncells <= 0 || nrecs <= 0) return cudaSuccess;
    PA_LAUNCH(blocks_for(ncells, 256), 256, 0, st, k_fp_unpack)(recs, nrecs, ncells, recv, pieces, scratch, ncrse, fboxes, flay, fbase, fcs, ncomp);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_fp_interp(bool conservative, const PaFpPiece* pieces, int npieces, long long ncells, const double* scratch,
                             long long ncrse, const int cdom_lo[3], const int cdom_hi[3], int ratio, const PaBoxDev* fboxes,
                             const PaLayDev* flay, double* fbase, long long fcs, int ncomp, cudaStream_t st) {
    if (ncells <= 0 || npieces <= 0) return cudaSuccess;
    Dom d;
    for (int a = 0; a < 3; ++a) { d.lo[a] = cdom_lo[a]; d.hi[a] = cdom_hi[a]; }
    if (conservative)
        PA_LAUNCH(blocks_for(ncells, 128), 128, 0, st, k_fp_interp<true>)(pieces, npieces, ncells, scratch, ncrse, d, ratio, fboxes, flay, fbase, fcs, ncomp);
    else
        PA_LAUNCH(blocks_for(ncells, 128), 128, 0, st, k_fp_interp<false>)(pieces, npieces, ncells, scratch, ncrse, d, ratio, fboxes, flay, fbase, fcs, ncomp);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_fp_clamp(const PaFpClamp* clamps, int nclamps, long long ncells, const int dom_lo[3], const int dom_hi[3], int g,
                            const PaBoxDev* boxes, const PaLayDev* lay, double* base, long long cs, int ncomp, cudaStream_t st) {
    if (ncells <= 0 || nclamps <= 0) return cudaSuccess;
    Dom d;
    for (int a = 0; a < 3; ++a) { d.lo[a] = dom_lo[a]; d.hi[a] = dom_hi[a]; }
    PA_LAUNCH(blocks_for(ncells, 256), 256, 0, st, k_fp_clamp)(clamps, nclamps, ncells, d, g, boxes, lay, base, cs, ncomp);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_filter(int g, const PaBoxDev* boxes, const PaLayDev* lin, const PaLayDev* lout, int nboxes, const long long* work_prefix,
                          long long nwork_per_comp, const double* in, long long cs_in, double* out, long long cs_out, int ncomp,
                          const double* w3_dev, cudaStream_t st) {
    if (nboxes <= 0 || nwork_per_comp <= 0 || ncomp <= 0) return cudaSuccess;
    const int W = 2 * g + 1;
    const size_t smem = (size_t)(W * W * W <= FILTER_MAX_W3 ? W * W * W : 0) * sizeof(double);
    const int grid = blocks_for(nwork_per_comp * ncomp, FILTER_THREADS, 148 * 64);
#define PA_FILTER_GO(GG) PA_LAUNCH(grid, FILTER_THREADS, smem, st, k_filter<GG>)(boxes, lin, lout, nboxes, work_prefix, in, cs_in, out, cs_out, ncomp, w3_dev, g)
    switch (g) {
    case 1: PA_FILTER_GO(1); break;
    case 2: PA_FILTER_GO(2); break;
    case 3: PA_FILTER_GO(3); break;
    case 4: PA_FILTER_GO(4); break;
    case 8: PA_FILTER_GO(8); break;
    default: PA_FILTER_GO(0); break;
    }
#undef PA_FILTER_GO
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace pa
