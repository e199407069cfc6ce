// kernels.cuh -- launch wrappers of the sm_100a kernels (definitions in kernels.cu / stencil_tma.cu).
#ifndef PA_KERNELS_CUH
#define PA_KERNELS_CUH

#include <cuda_runtime.h>

#include <atomic>

#include "pa_types.h"

// Kernel launch and dynamic shared memory, spelled as macros so that tests/emu can compile these same sources for its
// CPU emulation of the CUDA execution model (PA_HOST_EMULATION: a test-only build that checks indexing and the
// producer/consumer protocol without a GPU; it is never part of libpelestencil_b200.so and nothing in the product loads it).
#ifndef PA_HOST_EMULATION
#define PA_LAUNCH(grid, block, smem, stream, ...) __VA_ARGS__<<<(grid), (block), (smem), (stream)>>>
#define PA_DYN_SMEM(name) extern __shared__ __align__(128) unsigned char name[]
#endif

namespace pa {

// per-level device pointers handed to kernels by value
struct LevArgs {
    const PaBoxDev* boxes;      // boxes of the level, extended index (local boxes, then peer-owned link targets)
    const PaLayDev* lay_in;     // layout of the input field on this level (extended index)
    const PaLayDev* lay_out;    // layout of the output field
    const PaNbr* nbr;           // neighbour links of the local boxes
    const PaPeerSlab* peers;    // per rank: where that rank's slab of the INPUT field lives (comp 0 of the field)
    int in_comp;                // index of the first input component inside its field (peer slabs start at comp 0)
    const double* in;           // component 0 of the input field on this level
    double* out;                // component 0 of the output field
    long long cs_in, cs_out;    // component strides (elements)
    double dxi[3];              // 1/dx
};
struct GridArgs {
    LevArgs L[PA_MAX_LEVELS];
};

// stencil epilogues
enum StencilMode {
    MODE_GRAD = 0,      // in: 1 comp            out: gx, gy, gz, |g|                          (grad tool)
    MODE_GRAD3 = 1,     // in: 1 comp            out: gx, gy, gz                               (Hessian rows, velocity gradients)
    MODE_NORMAL = 2,    // in: c                 out: n = G/nrm (3 comps); aux out: G (3 comps) if aux != null
    MODE_DIV = 3,       // in: n (3 comps)       out: K = 0.5*(dnx/dx + dny/dy + dnz/dz), optional clip on c
    MODE_NORMAL_S = 4   // in: raw scalar S      out: n as MODE_NORMAL, plus Progress c = (S - pmin)*inv into cout[] --
                        // the progress pass fused into the loader.  Valid cells and linked neighbours hold S and are
                        // normalised on the fly; MATERIALISED ghost cells already hold c (see GhostXform)   (TMA kernel only)
};

// Ghost fill "in progress space" for MODE_NORMAL_S: the field holds the raw scalar S in its valid cells; every ghost
// cell the fill writes receives what the reference's Progress MultiFab would hold there -- a copied neighbour value is
// normalised on the way, and the Neumann / reflect_odd / coarse-fine formulas are evaluated on normalised inputs
// (curvature.cpp:310-322 then :447-457), so the results are bit-identical to normalise-then-fill.
struct GhostXform {
    int on;
    double pmin, inv;
};

struct StencilExtra {
    // MODE_NORMAL: optional un-normalised gradient output (the reference's cell_normal), per level, same layout as `out`
    double* aux[PA_MAX_LEVELS];
    long long cs_aux[PA_MAX_LEVELS];
    // MODE_DIV: optional threshold clip reading the progress variable (layout = lay_in)
    const double* prog[PA_MAX_LEVELS];
    int do_threshold;
    double threshold;
    // MODE_NORMAL_S / fused curvature: Progress output (one component, same layout as `out`) and the normalisation
    double* cout[PA_MAX_LEVELS];
    double pmin, inv;
    // fused curvature: MeanCurvature output (one component, same layout as `out`)
    double* kout[PA_MAX_LEVELS];
};

extern std::atomic<long long> g_launches;     // kernels launched by this library (host threads may launch concurrently)

// Every device allocation of the library goes through these two (api.cu), which keep the live bytes per device for
// pa_debug_device_bytes: a long series of plotfiles must not grow the device footprint.
cudaError_t dev_alloc(void** p, size_t bytes);
void dev_free(void* p);

cudaError_t launch_unpack_valid(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes,
                                long long ncells, const double* staging, double* comp_base, cudaStream_t st);
cudaError_t launch_pack_valid(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes,
                              long long ncells, const double* comp_base, double* staging, cudaStream_t st);
cudaError_t launch_fill(double* p, long long n, double v, cudaStream_t st);

// halo tags [tag0, tag1) covering cells [cell0, cell1) of the table's flattened enumeration; `comp0` = first component
// of the field being filled (peer slabs are addressed from the field's component 0)
cudaError_t launch_halo(const PaHaloTag* tags, int tag0, int tag1, long long cell0, long long cell1, const PaBoxDev* boxes,
                        const PaLayDev* lay, double* base, long long cs, int ncomp, const double* recv,
                        const PaPeerSlab* peers, int comp0, int rank, GhostXform xf, cudaStream_t st);
cudaError_t launch_exchange_pack(const PaPackTag* tags, long long tag0, long long tag1, long long dense0, long long ncells,
                                 const GridArgs& ga, int ncomp, double* send, cudaStream_t st);
// BC fill over the face chunks [blk0, blk1) (one thread block per chunk); coff = coarse gather offsets for the field's
// ghost width (Hier::crse_offsets)
cudaError_t launch_bcfill(const PaFaceRec* recs, const int* rec_level, const PaFaceBlock* blocks, long long blk0, long long blk1,
                          const unsigned short* flags, const long long* coff, const GridArgs& ga,
                          int ncomp, const double* recv, GhostXform xf, cudaStream_t st);

// stencils: GridArgs.in/out already point at the first component to read / write
cudaError_t launch_stencil_simple(int mode, const PaTile* tiles, int ntiles, const GridArgs& ga, const StencilExtra& ex,
                                  int nvar, cudaStream_t st);
// TMA-staged pipeline (cp.async.bulk + mbarrier ring, 2.5-D sweep along z).  max_plane_doubles / max_items = the largest staged
// plane (doubles, one component) and the largest number of x-pairs per plane over the given tiles (picks the CTA shape)
cudaError_t launch_stencil_tma(int mode, const PaTile* tiles, int ntiles, int max_plane_doubles, int max_items, const GridArgs& ga,
                               const StencilExtra& ex, int nvar, cudaStream_t st);
// device self-test: the branch-free sqrt / reciprocal / flame-normal forms of the TMA kernel against the plain operators on
// n pseudo-random operand sets; *bad_host = number of results that differ in any bit
cudaError_t selftest_math(long long n, unsigned long long seed, unsigned long long* bad_host, cudaStream_t st);
// Fused curvature (curv_fused.cu): S -> Progress, flame normal, and K on every cell whose K stencil stays inside its box.
// tiles: K rows / planes (subsets of [1, n-2]) of boxes at least 3 cells wide in every direction and at most
// curv_fused_max_nx() wide in x; GridArgs: in = S (nghost 1 layout), out = first flame-normal component; ex.cout / ex.kout /
// ex.aux / threshold as for the separate modes.
cudaError_t launch_curv_fused(const PaTile* tiles, int ntiles, int max_plane_doubles, const GridArgs& ga, const StencilExtra& ex,
                              bool plain_math, cudaStream_t st);
int curv_fused_consumer_warps();
int curv_fused_max_rows();           // staged rows per item (K rows + 4)
int curv_fused_max_plane_doubles();
// Third fused curvature kernel (curv_f3.cu, PA_CURV_FUSED=3): 256-thread CTAs, two per SM, one block barrier per plane.
// tiles: K rows (at most curv_f3_rows()) x K planes x an x strip; PaTile::lev = level | first K pair << 8 | K pairs << 16 with
// at most curv_f3_strip_pairs() pairs; boxes of even width >= 4, >= 3 cells in y and z.
// level_end[l] = number of tiles of levels 0 .. l (tiles are sorted by level; the kernel derives a CTA's level from blockIdx)
cudaError_t launch_curv_f3(const PaTile* tiles, int ntiles, const int* level_end, int nlev, const GridArgs& ga, const StencilExtra& ex,
                           cudaStream_t st);
int curv_f3_rows();
int curv_f3_strip_pairs();
// The same kernel without its K part (PA_NORMAL_F3=1): S -> Progress and n, the work of MODE_NORMAL_S.  tiles: rows (at most
// normal_f3_rows()) x planes x an x strip (at most normal_f3_strip_pairs() pairs) of whole boxes, strip encoded as above.
cudaError_t launch_normal_f3(const PaTile* tiles, int ntiles, const int* level_end, int nlev, const GridArgs& ga, const StencilExtra& ex,
                             cudaStream_t st);
int normal_f3_rows();
int normal_f3_strip_pairs();
// Barrier-free flame normal (normal_w.cu, PA_NORMAL_W=1): the work of MODE_NORMAL_S, one warp per row of an x strip, no shared
// memory.  tiles: at most normal_w_rows() rows x planes x a strip of 2 .. normal_w_strip_pairs() pairs, strip encoded as above.
cudaError_t launch_normal_w(const PaTile* tiles, int ntiles, const GridArgs& ga, const StencilExtra& ex, cudaStream_t st);
int normal_w_rows();
int normal_w_strip_pairs();
// K on the outermost cell layer of the boxes (the cells the fused kernel leaves out), from the ghost-filled flame normal:
// MODE_DIV's arithmetic, one thread per cell.  GridArgs: in = n (3 comps), out = K.
cudaError_t launch_div_shell(const int* box_level, const int* box_index, int nboxes, int blocks_per_box, const GridArgs& ga,
                             const StencilExtra& ex, cudaStream_t st);
// launch bookkeeping shared by the persistent kernels (stencil_tma.cu)
cudaError_t stencil_ticket(cudaStream_t st, unsigned long long nwork, int grid, unsigned long long** dev_out, unsigned long long* base_out);
int stencil_num_sms(cudaError_t* err);
int stencil_decide_normal_math(cudaStream_t st);   // 0 branch-free forms, 1 plain operators (runs the device self-test once)
void stencil_tma_release();      // frees the work-item ticket counters (pa_finalize)
int stencil_tma_normal_math();   // flame-normal arithmetic in use: 0 branch-free forms, 1 plain operators, -1 not decided yet
int stencil_tma_tile_rows();     // TY the tile table must be built with
int stencil_tma_max_tile_rows();
int stencil_tma_max_plane_doubles();

cudaError_t launch_field_hash(const PaBoxDev* boxes, const PaLayDev* lay, const int* gid, int nboxes, const double* base, long long cs,
                              int comp0, int ncomp, int lev, unsigned long long* out, cudaStream_t st);
cudaError_t launch_progress(const PaBoxDev* boxes, const PaLayDev* lay_in, const PaLayDev* lay_out, int nboxes,
                            const double* S, double* C, double pmin, double invdenom, cudaStream_t st);
cudaError_t launch_clip_normal(const PaBoxDev* boxes, const PaLayDev* lay_c, const PaLayDev* lay_n, int nboxes,
                               const double* C, double* N, long long cs_n, double thr, cudaStream_t st);
// pointwise Gaussian curvature from G (3), H (9), c -> Kg ; strain: div u from dU (9) ; velnormal
cudaError_t launch_gauss(const PaBoxDev* boxes, const PaLayDev* lay, const PaLayDev* lay_c, int nboxes, const double* G,
                         long long cs_g, const double* H, long long cs_h, const double* C, double* Kg, int do_thr,
                         double thr, cudaStream_t st);
cudaError_t launch_strain(const PaBoxDev* boxes, const PaLayDev* lay, int nboxes, const double* dU, long long cs,
                          double* sr, cudaStream_t st);
cudaError_t launch_velnormal(const PaBoxDev* boxes, const PaLayDev* lay_u, const PaLayDev* lay_n, const PaLayDev* lay_o,
                             int nboxes, const double* U, long long cs_u, const double* N, long long cs_n,
                             const double* C, double* out, int do_thr, double thr, cudaStream_t st);


// ---- filterPlt path (filter.cu) ----------------------------------------------------------------------------------------
// coarse valid cells -> coarse patches (scratch, component stride ncrse); pieces <- coarse patches (conservative linear with
// the mcslope limiter, or piecewise constant); ghost cells outside the domain <- clamped index; the filter itself
// same-level ghost copies, one thread block per (tag, slice of its rows / cells); local sources only (filterPlt path)
cudaError_t launch_halo_blocks(const PaHaloTag* tags, int ntags, int slices, const PaBoxDev* boxes, const PaLayDev* lay, double* base,
                               long long cs, int ncomp, cudaStream_t st);
cudaError_t launch_fp_gather(const PaFpCopy* copies, int ncopies, long long ncells, const PaFpPiece* pieces, const PaBoxDev* cboxes,
                             const PaLayDev* clay, const double* cbase, long long ccs, int ncomp, double* scratch, long long ncrse,
                             cudaStream_t st);
// several ranks: recv slab ([cell][comp]) -> ghost cells of local boxes and coarse-patch cells of the pieces
cudaError_t launch_fp_unpack(const PaFpUnpack* recs, int nrecs, long long ncells, const double* recv, const PaFpPiece* pieces,
                             double* scratch, long long ncrse, const PaBoxDev* fboxes, const PaLayDev* flay, double* fbase, long long fcs,
                             int ncomp, cudaStream_t st);
cudaError_t launch_fp_interp(bool conservative, const PaFpPiece* pieces, int npieces, long long ncells, const double* scratch,
                             long long ncrse, const int cdom_lo[3], const int cdom_hi[3], int ratio, const PaBoxDev* fboxes,
                             const PaLayDev* flay, double* fbase, long long fcs, int ncomp, cudaStream_t st);
cudaError_t launch_fp_clamp(const PaFpClamp* clamps, int nclamps, long long ncells, const int dom_lo[3], const int dom_hi[3], int g,
                            const PaBoxDev* boxes, const PaLayDev* lay, double* base, long long cs, int ncomp, cudaStream_t st);
// work_prefix: per box the prefix of (x-quads * row pairs * nz) = blocks of 4 x 2 cells, nboxes + 1 entries; w3_dev: (2g+1)^3 weight products, n slowest
cudaError_t launch_filter(int g, const PaBoxDev* boxes, const PaLayDev* lin, const PaLayDev* lout, int nboxes, const long long* work_prefix,
                          long long nwork_per_comp, const double* in, long long cs_in, double* out, long long cs_out, int ncomp,
                          const double* w3_dev, cudaStream_t st);
// ---- composite implicit-diffusion solve (smooth.cu) --------------------------------------------------------------------
// out = in - beta * Laplacian(in) on the valid cells of one level (`in` ghost-filled, one ghost layer)
cudaError_t launch_sm_apply(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                            const double* in, double* out, double beta, const double dxi[3], cudaStream_t st);
// out = rhs - A x on the valid cells of one level (`x` ghost-filled)
cudaError_t launch_sm_resid(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                            const double* rhs, const double* x, double* out, double beta, const double dxi[3], cudaStream_t st);
// one colour pass of red-black Gauss-Seidel on A x = rhs over one level (`x` ghost-filled): x += (rhs - A x) / diag on the valid
// cells with (i + j + k) mod 2 = colour
cudaError_t launch_sm_gsrb(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                           const double* rhs, double* x, double beta, const double dxi[3], double diag, int colour, cudaStream_t st);
// fine cells under the records' coarse cells += the coarse value (piecewise-constant prolongation)
cudaError_t launch_sm_prolong(const PaAvgDown* recs, int nrec, long long ncells, const PaBoxDev* cboxes, const PaLayDev* clay,
                              const PaBoxDev* fboxes, const PaLayDev* flay, const double* crse, double* fine, cudaStream_t st);
// coarse-fine faces of one (coarse level, dir, side) group: cout += the flux difference (average fine flux - coarse flux)
cudaError_t launch_sm_reflux(const PaReflux* recs, long long nrec, const PaLayDev* clay, const PaLayDev* flay, const double* cin,
                             const double* fin, double* cout, double beta, double dxic, double dxif, cudaStream_t st);
// covered cells of one coarse level <- average of their fine cells (or 0 when zero)
cudaError_t launch_sm_avgdown(const PaAvgDown* recs, int nrec, long long ncells, const PaBoxDev* cboxes, const PaLayDev* clay,
                              const PaBoxDev* fboxes, const PaLayDev* flay, double* crse, const double* fine, bool zero, cudaStream_t st);
// out = a*x + b*y + c*z elementwise over n doubles (y, z may be null)
cudaError_t launch_sm_lin3(long long n, double a, const double* x, double b, const double* y, double c, const double* z, double* out,
                           cudaStream_t st);
// partials of sum x*y (mode 0) or max |x| (mode 1) over the valid cells of one level -> partial[0 .. *nblocks)
cudaError_t launch_sm_reduce(const PaBoxDev* boxes, const PaLayDev* lay, const long long* host_off, int nboxes, long long ncells,
                             const double* x, const double* y, int mode, double* partial, int* nblocks, cudaStream_t st);
cudaError_t launch_sm_final(const double* partial, int n, int mode, double* out, cudaStream_t st);
int smooth_max_partials();            // most partials one launch_sm_reduce writes
// valid cells of one level, layout -> layout
cudaError_t launch_sm_copy(const PaBoxDev* boxes, const PaLayDev* lay_in, const PaLayDev* lay_out, const long long* host_off, int nboxes,
                           long long ncells, const double* in, double* out, cudaStream_t st);

// microbenchmark: blocks x threads threads each doing iters x 8 (multiply, add) pairs; out has blocks * threads doubles
cudaError_t launch_fp64_rate(double* out, int blocks, int threads, int iters, cudaStream_t st);

}  // namespace pa
#endif
