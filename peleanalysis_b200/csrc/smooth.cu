// smooth.cu -- kernels of the composite implicit-diffusion solve behind pa_smooth (curvature.cpp:328-406, do_smooth):
//     phi - beta * div(grad phi) = c   on the valid cells of every AMR level,
// the cell-centred 7-point operator with the ghost cells of the library's fill (same-level / periodic copies, wall rules,
// the coarse-fine polynomial), the coarse side of every coarse-fine face taking the average of the fine face fluxes
// (reflux), and covered coarse cells holding the average of their fine cells (average_down).  FP64 throughout; every
// reduction has a fixed order (per-thread strided partials, a block tree, one final block), so results do not depend on
// scheduling.  The host side (the Krylov loop) is in api.cu; DESIGN.md section 10 states the discrete system.
// Not a translation unit of its own: kernels.cu includes this file at its end (cell_addr, g_launches come from there).
#ifndef PA_SMOOTH_CU
#define PA_SMOOTH_CU

namespace pa {

namespace {

// valid cell number c of the level (local boxes in order, i fastest) -> box and box-relative (i, j, k)
__device__ __forceinline__ int sm_locate(const long long* __restrict__ host_off, int nboxes, const PaBoxDev* __restrict__ boxes,
                                         long long c, int& i, int& j, int& k) {
    int lo = 0, hi = nboxes;
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (host_off[mid] <= c) lo = mid; else hi = mid; }
    const PaBoxDev b = boxes[lo];
    const long long q = c - host_off[lo];
    i = (int)(q % b.n[0]);
    const long long r = q / b.n[0];
    j = (int)(r % b.n[1]);
    k = (int)(r / b.n[1]);
    return lo;
}

constexpr int SM_BLOCK = 256;
constexpr int SM_MAX_BLOCKS = 148 * 8;     // partials per level and reduction

int sm_grid(long long n) {
    long long g = (n + SM_BLOCK - 1) / SM_BLOCK;
    if (g > SM_MAX_BLOCKS) g = SM_MAX_BLOCKS;
    if (g < 1) g = 1;
    return (int)g;
}

// (A in)(a) = in - beta * sum_d ((in(+e_d) - in) * dxi_d - (in - in(-e_d)) * dxi_d) * dxi_d: the one expression of the operator,
// shared by its application, the residual and the Gauss-Seidel sweep
__device__ __forceinline__ double sm_op(const double* in, long long a, const PaLayDev& y, double beta, double dxi0, double dxi1,
                                        double dxi2) {
    const double v = in[a];
    const double lx = ((in[a + 1] - v) * dxi0 - (v - in[a - 1]) * dxi0) * dxi0;
    const double ly = ((in[a + y.P] - v) * dxi1 - (v - in[a - y.P]) * dxi1) * dxi1;
    const double lz = ((in[a + y.PS] - v) * dxi2 - (v - in[a - y.PS]) * dxi2) * dxi2;
    return v - beta * ((lx + ly) + lz);
}

// out = A in on every valid cell
__global__ void __launch_bounds__(SM_BLOCK) k_sm_apply(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay,
                                                     const long long* __restrict__ host_off, int nboxes, long long ncells,
                                                     const double* __restrict__ in, double* __restrict__ out, double beta,
                                                     double dxi0, double dxi1, double dxi2) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        int i, j, k;
        const int b = sm_locate(host_off, nboxes, boxes, c, i, j, k);
        const PaLayDev y = lay[b];
        const long long a = cell_addr(y, i, j, k);
        out[a] = sm_op(in, a, y, beta, dxi0, dxi1, dxi2);
    }
}

// out = rhs - A x on every valid cell
__global__ void __launch_bounds__(SM_BLOCK) k_sm_resid(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay,
                                                     const long long* __restrict__ host_off, int nboxes, long long ncells,
                                                     const double* __restrict__ rhs, const double* __restrict__ x,
                                                     double* __restrict__ out, double beta, double dxi0, double dxi1, double dxi2) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        int i, j, k;
        const int b = sm_locate(host_off, nboxes, boxes, c, i, j, k);
        const PaLayDev y = lay[b];
        const long long a = cell_addr(y, i, j, k);
        out[a] = rhs[a] - sm_op(x, a, y, beta, dxi0, dxi1, dxi2);
    }
}

// one colour of a red-black Gauss-Seidel sweep of A x = rhs: x += (rhs - A x) / diag on the valid cells with
// (i + j + k) mod 2 = colour in global level indices.  Such a cell reads only cells of the other colour inside its box, and
// ghost cells filled before the launch, so no cell is read and written in the same launch.
__global__ void __launch_bounds__(SM_BLOCK) k_sm_gsrb(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay,
                                                    const long long* __restrict__ host_off, int nboxes, long long ncells,
                                                    const double* __restrict__ rhs, double* x, double beta, double dxi0,
                                                    double dxi1, double dxi2, double diag, int colour) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        int i, j, k;
        const int b = sm_locate(host_off, nboxes, boxes, c, i, j, k);
        const PaBoxDev B = boxes[b];
        if (((B.lo[0] + i + B.lo[1] + j + B.lo[2] + k) & 1) != colour) continue;
        const PaLayDev y = lay[b];
        const long long a = cell_addr(y, i, j, k);
        x[a] += (rhs[a] - sm_op(x, a, y, beta, dxi0, dxi1, dxi2)) / diag;
    }
}

// coarse side of the coarse-fine faces of one (dir, side) group: every coarse cell appears at most once per launch
__global__ void __launch_bounds__(SM_BLOCK) k_sm_reflux(const PaReflux* __restrict__ recs, long long nrec,
                                                      const PaLayDev* __restrict__ clay, const PaLayDev* __restrict__ flay,
                                                      const double* __restrict__ cin, const double* __restrict__ fin,
                                                      double* __restrict__ cout, double beta, double dxic, double dxif) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nrec; q += (long long)gridDim.x * blockDim.x) {
        const PaReflux R = recs[q];
        const PaLayDev yc = clay[R.cbox], yf = flay[R.fbox];
        const int d = R.dir;
        const int t1 = (d == 0) ? 1 : 0, t2 = (d == 2) ? 1 : 2;
        const long long sc = (d == 0) ? 1 : (d == 1) ? (long long)yc.P : (long long)yc.PS;
        const long long sf = (d == 0) ? 1 : (d == 1) ? (long long)yf.P : (long long)yf.PS;
        const long long ac = cell_addr(yc, R.c[0], R.c[1], R.c[2]);
        const double F = R.side ? (cin[ac + sc] - cin[ac]) * dxic : (cin[ac] - cin[ac - sc]) * dxic;
        double g[4];
        for (int m = 0; m < 4; ++m) {
            int f[3] = {R.f[0], R.f[1], R.f[2]};
            f[t1] += m & 1; f[t2] += m >> 1;
            const long long af = cell_addr(yf, f[0], f[1], f[2]);
            // side 1: the fine region is above the coarse cell, its ghost cells below; side 0: the other way round
            g[m] = R.side ? (fin[af] - fin[af - sf]) * dxif : (fin[af + sf] - fin[af]) * dxif;
        }
        const double G = 0.25 * ((g[0] + g[1]) + (g[2] + g[3]));
        const double corr = beta * (G - F) * dxic;
        if (R.side) cout[ac] -= corr; else cout[ac] += corr;
    }
}

// covered coarse cells <- the average of their 8 fine cells (zero = false), or <- 0 (zero = true)
__global__ void __launch_bounds__(SM_BLOCK) k_sm_avgdown(const PaAvgDown* __restrict__ recs, int nrec, long long ncells,
                                                       const PaBoxDev* __restrict__ cboxes, const PaLayDev* __restrict__ clay,
                                                       const PaBoxDev* __restrict__ fboxes, const PaLayDev* __restrict__ flay,
                                                       double* __restrict__ crse, const double* __restrict__ fine, int zero) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        long long lo = 0, hi = nrec;
        while (hi - lo > 1) { long long mid = (lo + hi) >> 1; if (recs[mid].start <= c) lo = mid; else hi = mid; }
        const PaAvgDown R = recs[lo];
        const long long q = c - R.start;
        const int ci = R.lo[0] + (int)(q % R.n[0]);
        const long long r = q / R.n[0];
        const int cj = R.lo[1] + (int)(r % R.n[1]);
        const int ck = R.lo[2] + (int)(r / R.n[1]);
        const PaBoxDev cb = cboxes[R.cbox];
        double* p = crse + cell_addr(clay[R.cbox], ci - cb.lo[0], cj - cb.lo[1], ck - cb.lo[2]);
        if (zero) { *p = 0.0; continue; }
        const PaBoxDev fb = fboxes[R.fbox];
        const PaLayDev yf = flay[R.fbox];
        double s = 0.0;
        for (int kk = 0; kk < 2; ++kk)
            for (int jj = 0; jj < 2; ++jj)
                for (int ii = 0; ii < 2; ++ii)
                    s += fine[cell_addr(yf, 2 * ci + ii - fb.lo[0], 2 * cj + jj - fb.lo[1], 2 * ck + kk - fb.lo[2])];
        *p = 0.125 * s;
    }
}

// piecewise-constant prolongation over average-down records: each of the 8 fine cells of a record's coarse cell += the coarse value
__global__ void __launch_bounds__(SM_BLOCK) k_sm_prolong(const PaAvgDown* __restrict__ recs, int nrec, long long ncells,
                                                       const PaBoxDev* __restrict__ cboxes, const PaLayDev* __restrict__ clay,
                                                       const PaBoxDev* __restrict__ fboxes, const PaLayDev* __restrict__ flay,
                                                       const double* __restrict__ crse, double* __restrict__ fine) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        long long lo = 0, hi = nrec;
        while (hi - lo > 1) { long long mid = (lo + hi) >> 1; if (recs[mid].start <= c) lo = mid; else hi = mid; }
        const PaAvgDown R = recs[lo];
        const long long q = c - R.start;
        const int ci = R.lo[0] + (int)(q % R.n[0]);
        const long long r = q / R.n[0];
        const int cj = R.lo[1] + (int)(r % R.n[1]);
        const int ck = R.lo[2] + (int)(r / R.n[1]);
        const PaBoxDev cb = cboxes[R.cbox];
        const double v = crse[cell_addr(clay[R.cbox], ci - cb.lo[0], cj - cb.lo[1], ck - cb.lo[2])];
        const PaBoxDev fb = fboxes[R.fbox];
        const PaLayDev yf = flay[R.fbox];
        for (int kk = 0; kk < 2; ++kk)
            for (int jj = 0; jj < 2; ++jj)
                for (int ii = 0; ii < 2; ++ii)
                    fine[cell_addr(yf, 2 * ci + ii - fb.lo[0], 2 * cj + jj - fb.lo[1], 2 * ck + kk - fb.lo[2])] += v;
    }
}

// out = a*x + b*y + c*z over a whole level slab (valid cells, ghost cells and pads alike); y / z may be null
__global__ void __launch_bounds__(SM_BLOCK) k_sm_lin3(long long n, double a, const double* x, double b, const double* y, double c,
                                                    const double* z, double* out) {
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        double v = a * x[q];
        if (y) v += b * y[q];
        if (z) v += c * z[q];
        out[q] = v;
    }
}

// max that keeps a NaN (a NaN residual must never look converged)
__device__ __forceinline__ double sm_max(double m, double v) { return (v > m || v != v) ? v : m; }

// per-block partials over the valid cells of one level: mode 0 = sum x*y, mode 1 = max |x|
__global__ void __launch_bounds__(SM_BLOCK) k_sm_reduce(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay,
                                                      const long long* __restrict__ host_off, int nboxes, long long ncells,
                                                      const double* __restrict__ x, const double* __restrict__ y, int mode,
                                                      double* __restrict__ partial) {
    __shared__ double sh[SM_BLOCK];
    double acc = 0.0;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        int i, j, k;
        const int b = sm_locate(host_off, nboxes, boxes, c, i, j, k);
        const long long a = cell_addr(lay[b], i, j, k);
        if (mode == 0) acc += x[a] * y[a];
        else acc = sm_max(acc, fabs(x[a]));
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = SM_BLOCK / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] = (mode == 0) ? sh[threadIdx.x] + sh[threadIdx.x + s] : sm_max(sh[threadIdx.x], sh[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}

__global__ void __launch_bounds__(SM_BLOCK) k_sm_final(const double* __restrict__ partial, int n, int mode, double* __restrict__ out) {
    __shared__ double sh[SM_BLOCK];
    double acc = 0.0;
    for (int q = threadIdx.x; q < n; q += SM_BLOCK) acc = (mode == 0) ? acc + partial[q] : sm_max(acc, partial[q]);
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = SM_BLOCK / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] = (mode == 0) ? sh[threadIdx.x] + sh[threadIdx.x + s] : sm_max(sh[threadIdx.x], sh[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}

// valid cells of one level from one layout to another
__global__ void __launch_bounds__(SM_BLOCK) k_sm_copy(const PaBoxDev* __restrict__ boxes, const PaLayDev* __restrict__ lay_in,
                                                    const PaLayDev* __restrict__ lay_out, const long long* __restrict__ host_off,
                                                    int nboxes, long long ncells, const double* __restrict__ in,
                                                    double* __restrict__ out) {
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < ncells; c += (long long)gridDim.x * blockDim.x) {
        int i, j, k;
        const int b = sm_locate(host_off, nboxes, boxes, c, i, j, k);
        out[cell_addr(lay_out[b], i, j, k)] = in[cell_addr(lay_in[b], i, j, k)];
    }
}

}  // namespace

int smooth_max_partials() { return SM_MAX_BLOCKS; }

cudaError_t launch_sm_apply(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                            const double* in, double* out, double beta, const double dxi[3], cudaStream_t st) {
    if (ncells <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(ncells), SM_BLOCK, 0, st, k_sm_apply)(boxes, lay, host_off, nboxes, ncells, in, out, beta, dxi[0], dxi[1], dxi[2]);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_resid(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                            const double* rhs, const double* x, double* out, double beta, const double dxi[3], cudaStream_t st) {
    if (ncells <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(ncells), SM_BLOCK, 0, st, k_sm_resid)(boxes, lay, host_off, nboxes, ncells, rhs, x, out, beta, dxi[0], dxi[1], dxi[2]);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_gsrb(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                           const double* rhs, double* x, double beta, const double dxi[3], double diag, int colour, cudaStream_t st) {
    if (ncells <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(ncells), SM_BLOCK, 0, st, k_sm_gsrb)(boxes, lay, host_off, nboxes, ncells, rhs, x, beta, dxi[0], dxi[1], dxi[2], diag,
                                                           colour);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_prolong(const PaAvgDown* recs, int nrec, long long ncells, const PaBoxDev* cboxes, const PaLayDev* clay,
                              const PaBoxDev* fboxes, const PaLayDev* flay, const double* crse, double* fine, cudaStream_t st) {
    if (ncells <= 0 || nrec <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(ncells), SM_BLOCK, 0, st, k_sm_prolong)(recs, nrec, ncells, cboxes, clay, fboxes, flay, crse, fine);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_reflux(const PaReflux* recs, long long nrec, const PaLayDev* clay, const PaLayDev* flay, const double* cin,
                             const double* fin, double* cout, double beta, double dxic, double dxif, cudaStream_t st) {
    if (nrec <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(nrec), SM_BLOCK, 0, st, k_sm_reflux)(recs, nrec, clay, flay, cin, fin, cout, beta, dxic, dxif);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_avgdown(const PaAvgDown* recs, int nrec, long long ncells, const PaBoxDev* cboxes, const PaLayDev* clay,
                              const PaBoxDev* fboxes, const PaLayDev* flay, double* crse, const double* fine, bool zero, cudaStream_t st) {
    if (ncells <= 0 || nrec <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(ncells), SM_BLOCK, 0, st, k_sm_avgdown)(recs, nrec, ncells, cboxes, clay, fboxes, flay, crse, fine, zero ? 1 : 0);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_lin3(long long n, double a, const double* x, double b, const double* y, double c, const double* z, double* out,
                           cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(n), SM_BLOCK, 0, st, k_sm_lin3)(n, a, x, b, y, c, z, out);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_reduce(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                             const double* x, const double* y, int mode, double* partial, int* nblocks, cudaStream_t st) {
    *nblocks = 0;
    if (ncells <= 0) return cudaSuccess;
    const int g = sm_grid(ncells);
    PA_LAUNCH(g, SM_BLOCK, 0, st, k_sm_reduce)(boxes, lay, host_off, nboxes, ncells, x, y, mode, partial);
    ++g_launches;
    *nblocks = g;
    return cudaGetLastError();
}

cudaError_t launch_sm_final(const double* partial, int n, int mode, double* out, cudaStream_t st) {
    PA_LAUNCH(1, SM_BLOCK, 0, st, k_sm_final)(partial, n, mode, out);
    ++g_launches;
    return cudaGetLastError();
}

cudaError_t launch_sm_copy(const PaBoxDev* boxes, const PaLayDev* lay_in, const PaLayDev* lay_out, const long long* host_off, int nboxes,
                           long long ncells, const double* in, double* out, cudaStream_t st) {
    if (ncells <= 0) return cudaSuccess;
    PA_LAUNCH(sm_grid(ncells), SM_BLOCK, 0, st, k_sm_copy)(boxes, lay_in, lay_out, host_off, nboxes, ncells, in, out);
    ++g_launches;
    return cudaGetLastError();
}

}  // namespace pa

#endif  // PA_SMOOTH_CU
