/* pele_stencil_b200.h -- C ABI of the B200-native derived-field stencil path of PeleAnalysis
 * (ghost-cell fill -> centred-difference gradient / mean curvature, per FAB, per AMR level).
 *
 * The library replaces, for this path only, the AMReX C++ objects the reference tools drive between
 * "data is in state[lev]" (Src/grad.cpp:167, Src/curvature.cpp:305) and WriteMultiLevelPlotfile
 * (Src/grad.cpp:256, Src/curvature.cpp:843).  Each entry point cites the reference interface it stands
 * in for (AX/ = Submodules/PelePhysics/Submodules/amrex/Src/).  INTEGRATION.md shows the call sequence a
 * maintainer adds to grad.cpp / curvature.cpp.
 *
 * Conventions: extern "C"; plain pointers and sizes; every function returns 0 on success or a negative
 * pa_status and never throws; pa_last_error() returns a thread-local message.  The library owns all device
 * memory.  One host thread drives one pa_hier.  There is NO CPU fallback: compute entry points fail with
 * PA_ERR_CUDA when no sm_100 device is usable.
 *
 * Host buffers are FArrayBox-ordered: the VALID region of one box, one component, i fastest
 * ([nz][ny][nx] doubles) -- what FArrayBox::dataPtr(comp) addresses for a 0-ghost FAB.
 */
#ifndef PELE_STENCIL_B200_H
#define PELE_STENCIL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    PA_OK = 0,
    PA_ERR_ARG = -1,        /* bad argument / inconsistent hierarchy (message says which) */
    PA_ERR_CUDA = -2,       /* CUDA runtime error or no usable device */
    PA_ERR_NOMEM = -3,
    PA_ERR_UNSUPPORTED = -4,
    PA_ERR_STATE = -5,      /* call order (e.g. remote halo data not exchanged yet) */
    PA_ERR_NOCONV = -6      /* an iterative solve did not converge (pa_last_error gives the residual reached) */
} pa_status;

/* Domain-boundary kinds for NON-periodic directions: LinOpBCType::Neumann / reflect_odd as chosen by the
 * tools from is_per / sym_dir (Src/grad.cpp:182-193, Src/curvature.cpp:429-441). */
enum { PA_BC_NEUMANN = 0, PA_BC_REFLECT_ODD = 1 };

/* One AMR level: Geometry + BoxArray + DistributionMapping (Src/grad.cpp:160-164). */
typedef struct {
    int domain_lo[3], domain_hi[3];   /* AmrData::ProbDomain()[lev], inclusive cell indices */
    double dx[3];                     /* Geometry::CellSize(): (prob_hi-prob_lo)/N, AX/Base/AMReX_Geometry.cpp:520 */
    int nboxes;
    const int *boxes;                 /* nboxes x 6: lo[3], hi[3] (BoxArray) */
    const int *owner;                 /* nboxes ranks (DistributionMapping) or NULL = everything on rank 0 */
} pa_level_desc;

typedef struct pa_hier pa_hier;
typedef struct pa_field pa_field;

/* Options of the curvature tool (ParmParse keys of Src/curvature.cpp:72-106). */
typedef struct {
    double prog_min, prog_max;        /* progMin / progMax (after the file min/max reduction) */
    int do_threshold;                 /* threshold_prog */
    double threshold;                 /* threshold_value */
    int do_gauss;                     /* do_gaussCurv */
    int do_strain;                    /* do_strain (StrainRate = div u, reproducing the reference's overwrite at :736-747) */
    int get_strain_tensor;            /* getStrainTensor */
    int do_velnormal;                 /* do_velnormal */
    int reserved[8];
} pa_curv_opts;

/* Options of curvature's do_smooth (ParmParse smoothing_time of Src/curvature.cpp:72-106; the solve of :328-406). */
typedef struct {
    double smoothing_time;            /* smoothing_time: beta of phi - beta * div(grad phi) = c (>= 0) */
    double tol_rel;                   /* stop when max|c - A phi| <= tol_rel * max|c| over uncovered cells; 0 = 1e-10 */
    int max_iter;                     /* iterations before PA_ERR_NOCONV; 0 = 1000 */
    int precond;                      /* preconditioner of the solve: PA_SMOOTH_PRECOND_* (0 = Jacobi) */
    int reserved[7];
} pa_smooth_opts;
enum {
    PA_SMOOTH_PRECOND_JACOBI = 0,     /* per-level inverse diagonal */
    PA_SMOOTH_PRECOND_MG = 1          /* one multigrid V-cycle (red-black Gauss-Seidel, composite restriction; see pa_smooth) */
};

/* ---- runtime ------------------------------------------------------------------------------------- */
/* Select the CUDA device of this process (one process per GPU).  amrex::Initialize's device part. */
int pa_init(int device);
int pa_finalize(void);
const char *pa_last_error(void);
const char *pa_version(void);
/* Stream all subsequent work of this thread's library calls is enqueued on (a cudaStream_t; NULL = default). */
int pa_set_stream(void *cuda_stream);
int pa_sync(void);                     /* cudaStreamSynchronize on that stream */
/* Pinned host memory for upload/download buffers (cudaHostAlloc / cudaFreeHost). */
int pa_host_alloc(void **p, size_t bytes);
int pa_host_free(void *p);
int pa_host_register(void *p, size_t bytes);   /* pin caller-owned memory, e.g. FArrayBox storage */
int pa_host_unregister(void *p);

/* ---- hierarchy: replaces MLPoisson(geoms,grids,dmaps,info) + setMaxOrder(4) + setDomainBC(lo,hi) ----
 * (Src/grad.cpp:173-193; AX/LinearSolvers/MLMG/AMReX_MLCellLinOp.H:368-509 defineAuxData/defineBC).
 * Builds, on the host, the copy-descriptor tables the device kernels consume: same-level/periodic halo rows
 * (FabArrayBase::FB, AX/Base/AMReX_FabArrayBase.cpp:658-877), face masks (AX/Boundary/AMReX_MultiMask.cpp:25-71),
 * box-face BC records (AX/LinearSolvers/MLMG/AMReX_MLMGBndry.H:107-155) and the coarse gather index of every
 * coarse-fine face (BndryRegister, AX/Boundary/AMReX_BndryRegister.H:147-190,266-276).
 * The refinement ratio of each level is taken from the level domains (AX/LinearSolvers/MLMG/AMReX_MLLinOp.H:856-885).
 * rank / nranks: this process and the number of processes the boxes are distributed over (owner[] values). */
int pa_hier_create(pa_hier **h, int nlev, const pa_level_desc *levels, const int is_per[3],
                   const int bc_kind[3], int rank, int nranks);
/* The same with flags.  By default every box face whose whole ghost layer lies inside ONE same-level box of equal
 * x/y extent on the same rank gets a "neighbour link": the stencil kernels read the neighbour's valid cells in place
 * (TMA bulk copies / scalar loads) and those ghost cells are never materialised -- the FillBoundary traffic of
 * AX/Base/AMReX_FBI.H:211-267 disappears for them.  pa_fill_ghosts / pa_fill_boundary still materialise everything.
 *   PA_HIER_PEER_LINKS  links may also point at boxes of OTHER ranks; their slabs are then read over NVLink through
 *                       CUDA-IPC mappings (pa_field_ipc_handle / pa_field_map_peer), replacing the MPI send/recv of
 *                       AX/Base/AMReX_FabArrayCommI.H:62-110 for those faces.
 *   PA_HIER_NO_LINKS    no links at all: every ghost cell is materialised by the halo gather (reference data flow).
 *   PA_HIER_FILTER_ONLY grids of the filterPlt path (pa_fill_patch / pa_filter): BoxArray::maxSize may cut fine boxes at
 *                       positions that are not multiples of the refinement ratio, which FillPatch accepts and MLMG's
 *                       coarse-fine stencil does not.  No face masks / BC records are built; pa_grad, pa_curvature and
 *                       pa_fill_ghosts return PA_ERR_UNSUPPORTED on such a hierarchy. */
enum { PA_HIER_PEER_LINKS = 1, PA_HIER_NO_LINKS = 2, PA_HIER_FILTER_ONLY = 4 };
int pa_hier_create2(pa_hier **h, int nlev, const pa_level_desc *levels, const int is_per[3],
                    const int bc_kind[3], int rank, int nranks, unsigned flags);
int pa_hier_destroy(pa_hier *h);
int pa_hier_num_levels(const pa_hier *h);
int pa_hier_num_boxes(const pa_hier *h, int lev);          /* global count */
int64_t pa_hier_num_cells(const pa_hier *h, int lev);      /* valid cells, global; lev<0 = all levels */
int64_t pa_hier_num_local_cells(const pa_hier *h, int lev);
int pa_hier_box_owner(const pa_hier *h, int lev, int box);

/* Morton/SFC box -> rank map balanced by cell count (DistributionMapping default strategy,
 * AX/Base/AMReX_DistributionMapping.cpp:42,1262-1320).  owner_out has nboxes entries. */
int pa_sfc_distribute(int nboxes, const int *boxes, int nranks, int *owner_out);

/* ---- device MultiFab: replaces MultiFab(ba, dm, ncomp, nghost) (Src/grad.cpp:164) ------------------ */
int pa_field_alloc(pa_hier *h, int ncomp, int nghost, pa_field **f);
int pa_field_free(pa_field *f);
int pa_field_ncomp(const pa_field *f);
int pa_field_nghost(const pa_field *f);
int64_t pa_field_bytes(const pa_field *f);
/* Peer mapping for PA_HIER_PEER_LINKS hierarchies (one process per GPU on one NVLink node).  Each rank exports a
 * 64-byte cudaIpcMemHandle_t per level (all zero if it owns no box there), the caller moves the handles between the
 * processes (MPI_Allgather / torch.distributed.all_gather), and every rank maps the others'.  The caller must also
 * order the peers' writes before this rank's reads (a barrier after uploads / between dependent passes). */
int pa_field_ipc_handle(const pa_field *f, int lev, void *handle64);
int pa_field_map_peer(pa_field *f, int lev, int peer_rank, const void *handle64);
/* Valid region of one (level, box, comp) <-> host, asynchronous on the library stream.  Stands in for the
 * FillVar copy into state[lev] (Src/grad.cpp:167) and the ghost-stripping copy before VisMF::Write
 * (AX/Base/AMReX_PlotFileUtil.cpp:227-233).  Boxes owned by other ranks are rejected with PA_ERR_ARG. */
int pa_field_upload(pa_field *f, int lev, int box, int comp, const double *host_valid);
int pa_field_download(const pa_field *f, int lev, int box, int comp, double *host_valid);
/* Whole level at once: host buffer = this rank's boxes of the level concatenated in box order (each [nz][ny][nx]). */
int pa_field_upload_level(pa_field *f, int lev, int comp, const double *host_concat);
int pa_field_download_level(const pa_field *f, int lev, int comp, double *host_concat);
int pa_field_set_val(pa_field *f, int comp, int ncomp, double v);     /* MultiFab::setVal incl. ghost cells */
/* Fingerprint of the valid cells of comps [comp, comp+ncomp) of this rank's boxes: sum mod 2^64 of a mix of every cell's bit
 * pattern with (level, GLOBAL box id, component, cell index).  Adding the ranks' values (wrapping) gives a number that does
 * not depend on the box -> rank map: equal fingerprints for 1, 2, 4, 8 ranks <=> bit-identical outputs (with overwhelming
 * probability).  Synchronises the stream.  No reference counterpart (the nearest is MultiFab::sum, AMReX_MultiFab.H). */
int pa_field_hash(const pa_field *f, int comp, int ncomp, uint64_t *out);

/* ---- ghost cells ------------------------------------------------------------------------------------ */
/* FabArray::FillBoundary(scomp, ncomp, periodicity, cross) (AX/Base/AMReX_FabArrayCommI.H:7-60): same-level and
 * periodic copies into all nghost layers; cross!=0 fills only the width-1 face layers a cross stencil reads. */
int pa_fill_boundary(pa_field *f, int comp, int ncomp, int cross);
/* MLCellLinOp::applyBC in inhomogeneous mode with coarse data (AX/LinearSolvers/MLMG/AMReX_MLCellLinOp.H:680-889)
 * = FillBoundary(cross) + coarse-fine o3 interpolation (AX/Boundary/AMReX_InterpBndryData_3D_K.H:23-119) +
 * mllinop_apply_bc (AX/LinearSolvers/MLMG/AMReX_MLLinOp_K.H:14-325) on every level in [lev_lo, lev_hi].
 * Coarse values are the VALID cells of the same component on level-1 (what updateSolBC/setCoarseFineBC pass). */
int pa_fill_ghosts(pa_field *f, int comp, int ncomp, int lev_lo, int lev_hi);

/* ---- the two tools' hot paths ------------------------------------------------------------------------ */
/* grad: for v in [0,nvar): (gx,gy,gz,|g|) of in[comp_in+v] -> out[comp_out+4v .. +3]; includes the ghost fill.
 * Replaces Src/grad.cpp:169-236 (FillBoundary, setLevelBC, MLMG::apply, MLMG::getFluxes,
 * average_face_to_cellcenter, mult(-1), magnitude lambda).  `in` needs nghost>=1. */
int pa_grad(pa_field *in, int comp_in, int nvar, pa_field *out, int comp_out);
/* The same in two separately callable phases, so a caller can time (or overlap) them: phases bit 0 = ghost fill
 * (halo gather + coarse-fine / wall fill), bit 1 = stencil sweep.  pa_grad == pa_grad_phases(..., 3). */
int pa_grad_phases(pa_field *in, int comp_in, int nvar, pa_field *out, int comp_out, int phases);
/* curvature: S = state[comp_S]; writes Progress, MeanCurvature, FlameNormalX/Y/Z into out[comp_out..+4], then
 * (if enabled, in this order) GaussianCurvature, StrainRate, 9 ROST comps, VelFlameNormal.
 * Velocities (do_strain / do_velnormal) are state[comp_vel..+2].  Replaces Src/curvature.cpp:310-326,418-791.
 * `state` needs nghost>=1 (nghost == 1 selects the fused TMA kernels); `out` must have nghost == 1 (Progress and the flame
 * normal are ghost-filled in place). */
int pa_curvature(pa_field *state, int comp_S, int comp_vel, const pa_curv_opts *opts, pa_field *out, int comp_out);
int pa_curvature_num_outputs(const pa_curv_opts *opts);
/* The same in its two passes, so a multi-rank caller can put the cross-rank step between them (the reference does the
 * same thing with MPI inside FillBoundary / ParallelCopy of the flame normal, Src/curvature.cpp:487-502,514-520):
 *   phases bit 0: progress variable + ghost fill of S + flame normal (writes Progress, FlameNormalX/Y/Z);
 *                 multi-rank: the caller has exchanged state[comp_S] (pa_exchange_pack -> transport -> mark_received)
 *   phases bit 1: ghost fill of the normal + MeanCurvature + the optional branches;
 *                 multi-rank: the caller has exchanged out[comp_out+2 .. +4], and with peer links has ordered every
 *                 rank's pass 1 before this call (a cross-rank barrier on the stream).
 * pa_curvature == pa_curvature_phases(..., 3) and is single-rank only.  On multi-rank hierarchies the two phases cover the
 * default options and do_velnormal; threshold_prog / do_gaussCurv / do_strain need further cross-rank steps and return
 * PA_ERR_UNSUPPORTED here -- use pa_curvature_steps for those (every option is supported there). */
int pa_curvature_phases(pa_field *state, int comp_S, int comp_vel, const pa_curv_opts *opts, pa_field *out, int comp_out,
                        int phases);

/* The same as single steps, for multi-rank callers whose options need more cross-rank steps than the two passes above
 * (threshold_prog: the flame normal is exchanged before EVERY level's divergence, because level l reads the clipped
 * normal of level l-1, Src/curvature.cpp:514-518 after :549-567; do_gaussCurv: the un-normalised gradient, an internal
 * field, is exchanged too, :575-612; do_strain: the velocities, :686-717).  `steps` is a combination of PA_CURV_*; the
 * level range applies to PA_CURV_DIV and PA_CURV_CLIP only (-1, -1 = all levels).  Before each step the caller has exchanged
 * what it reads:
 *   PA_CURV_PASS1  state[comp_S]          PA_CURV_DIV    out[comp_out+2 .. +4]  (with threshold_prog: one level per call)
 *   PA_CURV_GAUSS  scratch field 0 (3)    PA_CURV_STRAIN state[comp_vel .. +2]  PA_CURV_VELN   nothing
 *   PA_CURV_CLIP   nothing -- but it zeroes the flame normal of the level IN PLACE where the progress variable is outside
 *                  [threshold, 1-threshold] (:549-567), and PA_CURV_DIV of the same level reads the UNCLIPPED normal of other
 *                  boxes (on a peer-linked hierarchy: of other ranks, in place): a multi-rank caller puts a cross-rank
 *                  barrier between DIV(l) and CLIP(l), and the exchange / barrier for level l+1 after CLIP(l).  Without
 *                  threshold_prog the step does nothing.  Single-rank: DIV | CLIP in one call runs them level by level.
 * pa_curvature_phases(1) == PA_CURV_PASS1, (2) == all the other steps. */
enum { PA_CURV_PASS1 = 1, PA_CURV_DIV = 2, PA_CURV_GAUSS = 4, PA_CURV_STRAIN = 8, PA_CURV_VELN = 16, PA_CURV_CLIP = 32 };
int pa_curvature_steps(pa_field *state, int comp_S, int comp_vel, const pa_curv_opts *opts, pa_field *out, int comp_out,
                       int steps, int lev_lo, int lev_hi);
/* Internal field a multi-rank caller must exchange / peer-map: which = 0, the un-normalised gradient of the progress
 * variable (3 components, nghost 1).  Owned by the hierarchy; do not free. */
int pa_curvature_scratch(pa_hier *h, int which, pa_field **f);

/* ---- do_smooth: one backward-Euler diffusion step of the progress variable (Src/curvature.cpp:328-406) ----------------------
 * The reference builds MLABecLaplacian(alpha = 1, a = 1, beta = smoothing_time, b = 1) on all levels and MLMG-solves
 *     phi - beta * div(grad phi) = c,   c = (S - prog_min) / (prog_max - prog_min),
 * as one composite AMR system: the 7-point operator on every valid cell with the ghost cells of pa_fill_ghosts (same-level /
 * periodic copies, Neumann / reflect_odd walls, the coarse-fine polynomial through the o3-interpolated coarse value, here of
 * maxorder 3), the coarse side of every coarse-fine face taking the average of the fine face fluxes, covered coarse cells holding
 * the average of their fine cells.  Writes c into out[comp_c] -- bit-identical to pa_curvature's Progress -- and phi into
 * out[comp_phi]; the curvature of the smoothed field is then pa_curvature on phi with prog_min = 0, prog_max = 1.
 * Solver: right-preconditioned BiCGStab on the composite residual, deterministic (fixed reduction order); the stop test is on
 * the TRUE residual.  *iters = iterations, *resid = max|c - A phi| / max|c| over uncovered cells (both may be NULL).
 * Preconditioner (o->precond): PA_SMOOTH_PRECOND_JACOBI, the inverse diagonal of each level's operator, whose iteration count
 * grows with smoothing_time / dx_finest^2; or PA_SMOOTH_PRECOND_MG, one V-cycle per application: red-black Gauss-Seidel on the
 * AMR levels from the finest down, the composite residual restricted level by level, a geometric V-cycle over level 0's own
 * coarsenings by 2 (as far as every box of level 0 coarsens), then back up with piecewise-constant prolongation.  The
 * V-cycle is a fixed linear map (fixed sweep counts), so runs stay bit-identical; the discrete system, the stop test, the
 * restarts and every error code are the same in both modes.  Another precond value: PA_ERR_ARG.
 * smoothing_time = 0 copies c into phi bit for bit.  One rank and refinement ratio 2 only (PA_ERR_UNSUPPORTED otherwise);
 * negative smoothing_time: PA_ERR_ARG; not converged within max_iter: PA_ERR_NOCONV, phi not written. */
int pa_smooth(pa_field *state, int comp_S, double prog_min, double prog_max, const pa_smooth_opts *o, pa_field *out, int comp_c,
              int comp_phi, int *iters, double *resid);

/* ---- filterPlt: the neighbouring stencil tool (Src/filterPlt.cpp:100-222; SURVEY 8(f) rank 4) -------------------------
 * PP/ = Submodules/PelePhysics/Source.  The tool re-chops the plotfile's grids to max_grid_size, fills nGrow = fgr/2 ghost
 * layers of every level by FillPatch rules on a NON-periodic geometry (PP/Utility/PltFileManager/PltFileManager.cpp:118-120)
 * and applies PelePhysics' Filter box by box.  Create the hierarchy with is_per = {0,0,0} on the re-chopped grids, allocate the
 * input field with nghost >= the widest level's nGrow and upload the plotfile's valid data; then per level
 * pa_fill_patch + pa_filter.  Results are bit-identical to the reference tool's.  On several ranks (boxes of every level
 * distributed, e.g. by pa_sfc_distribute) each pa_fill_patch is preceded by its exchange, below. */
/* Filter::Filter(type, fgr) (PP/Utility/Filter/Filter.H:56-111 + Filter.cpp:3-404): ghost width and the 2*ngrow+1 weights of
 * filter_types 0..10 (1 box, 2 Gaussian, 3-10 the Sagaut & Grohens approximations).  Returns the number of weights
 * (weights may be NULL to query) or a negative pa_status. */
int pa_filter_weights(int filter_type, int fgr, int *ngrow, double *weights, int cap);
/* BoxArray::maxSize(max_grid_size) (AX/Base/AMReX_BoxArray.cpp:549-564 -> AMReX_BoxList.cpp:765-815) on nboxes x 6 ints:
 * every box replaced, in place, by its chunks.  Returns the new box count (out_boxes may be NULL to query). */
int pa_boxes_max_size(int nboxes, const int *boxes, int max_grid_size, int *out_boxes, int cap);
/* Ghost cells of level `lev`, `nghost` layers, as Src/filterPlt.cpp:170-203 fills them: FillPatchSingleLevel on level 0,
 * FillPatchTwoLevels above (AX/AmrCore/AMReX_FillPatchUtil_I.H) -- same-level valid data where a box of the level covers the
 * cell; else interpolation from the VALID cells of level lev-1 (interp_type 1: MFCellConsLinInterp with the monotonised-central
 * slope, AX/AmrCore/AMReX_MFInterp_3D_C.H:178-260; 0: MFPCInterp); first-order extrapolation outside the domain
 * (AX/Base/AMReX_PhysBCFunct.H:406-640, AMReX_FilCC_3D_C.H), on the coarse patch as well.  Levels are independent of each
 * other (only valid coarse data is read).  PA_ERR_ARG if the coarse level does not cover a needed coarse patch (decided over
 * every box of the level: on several ranks all fail or none does), or, on several ranks, if this rank receives cells for the
 * fill and the recv slab was not marked for exactly this (field, comp, ncomp, lev, nghost, interp_type). */
int pa_fill_patch(pa_field *f, int comp, int ncomp, int lev, int nghost, int interp_type);
/* Several ranks: the communication of FabArray::FillPatchTwoLevels (ParallelCopy of the coarse patches and FillBoundary of
 * the fine level, AX/AmrCore/AMReX_FillPatchUtil_I.H; AX/Base/AMReX_FabArrayCommI.H) as one packed-slab exchange per fill:
 *   pa_fill_patch_pack -> transport (NCCL send/recv or pa_copy_async of each peer's segment) -> pa_fill_patch_mark_received
 *   -> pa_fill_patch
 * Sources owned by another rank than their destination box's -- same-level neighbours and coarse cells of the patches --
 * travel [cell][comp] in doubles; offsets (nranks+1 each) locate each peer's segment.  The slabs are shared by every fill
 * of the hierarchy and grow to the largest plan asked for: query the buffers again after asking for another plan.  Any pack
 * invalidates the mark of the previous fill.  On one rank the offsets are all zero, the slabs NULL and pack / mark do
 * nothing, so callers need a single code path. */
int pa_fill_patch_exchange_buffers(pa_field *f, int ncomp, int lev, int nghost, int interp_type, double **send_slab, double **recv_slab,
                                   int64_t *send_offsets /*nranks+1*/, int64_t *recv_offsets /*nranks+1*/);
int pa_fill_patch_pack(pa_field *f, int comp, int ncomp, int lev, int nghost, int interp_type);
int pa_fill_patch_mark_received(pa_field *f, int comp, int ncomp, int lev, int nghost, int interp_type);
/* Filter::apply_filter on every box of level `lev` (PP/Utility/Filter/Filter.H:28-50, Filter.cpp:462-491):
 * out = sum over (n, m, l) of w[l]*w[m]*w[n] * in(i+l, j+m, k+n), the reference's summation order.  `in` must hold ngrow
 * filled ghost layers (pa_fill_patch); out's ghost cells are not written. */
int pa_filter(pa_field *in, int comp_in, pa_field *out, int comp_out, int ncomp, int lev, int filter_type, int fgr);
/* ---- ranks that share ONE process (one host thread per GPU, e.g. an OpenMP-style host without MPI) -------------------
 * The calling thread's GPU is the one its pa_init named.  pa_enable_peer_access lets that GPU address a peer GPU's memory
 * (cudaDeviceEnablePeerAccess); pa_field_slab gives the level slab a peer thread passes to pa_field_map_peer_ptr -- the
 * same-address-space form of pa_field_ipc_handle / pa_field_map_peer; pa_copy_async is a device-to-device copy on the
 * calling thread's stream that may cross GPUs (it moves a peer's send slab segment into this rank's recv slab).
 * Together they stand where the reference has its MPI layer under FillBoundary / ParallelCopy
 * (AX/Base/AMReX_FabArrayCommI.H:7-60 FBEP_nowait / FillBoundary_finish, AX/Base/AMReX_ParallelDescriptor.H). */
int pa_enable_peer_access(int peer_device);
int pa_field_slab(const pa_field *f, int lev, const double **base);
int pa_field_map_peer_ptr(pa_field *f, int lev, int peer_rank, const double *base);
int pa_copy_async(double *dst, const double *src, int64_t n);

/* ---- multi-rank ghost exchange (one process per GPU; the transport is the caller's: NCCL send/recv) ---
 * For exchange step `step` of an operation the library packs what each peer needs into a device send slab and
 * unpacks the peer's slab after the caller moved it.  Sizes are in doubles.  Single-rank hierarchies have
 * zero-length slabs and never need these calls. */
int pa_exchange_counts(const pa_hier *h, int nghost, int ncomp, int64_t *send_counts /*nranks*/, int64_t *recv_counts /*nranks*/);
int pa_exchange_buffers(pa_field *f, int ncomp, double **send_slab, double **recv_slab,
                        int64_t *send_offsets /*nranks+1*/, int64_t *recv_offsets /*nranks+1*/);
int pa_exchange_pack(pa_field *f, int comp, int ncomp);     /* valid cells peers need -> send slab */
int pa_exchange_mark_received(pa_field *f, int comp, int ncomp);   /* recv slab now holds the peers' data */
/* Split grad so the caller can exchange between the phases: pack (above) -> [transport] -> pa_grad. */

/* ---- instrumentation --------------------------------------------------------------------------------- */
int64_t pa_kernel_launches(void);              /* number of kernels this library launched so far (this process) */
/* Bytes of device memory the library holds on the calling thread's current device: every live allocation of hierarchies,
 * fields and the library's internal counters.  After a hierarchy and its fields are freed, only the per-stream counters
 * the first kernels created remain, so the value returns to the same number after every file of a series. */
int pa_debug_device_bytes(int64_t *out);
int pa_hier_build_seconds(const pa_hier *h, double *seconds);
/* Algorithmic bytes of SURVEY 8(d): sum over local boxes of 8*V_in + 8*nout*V, V_in = V + 2(nx*ny+ny*nz+nx*nz). */
int64_t pa_algorithmic_bytes(const pa_hier *h, int nout_per_cell);

/* ---- debug / parity inspection (integer tables are compared bit-exactly with the oracle) ------------- */
/* A (level, box, comp) including its ghost cells, [nz+2g][ny+2g][nx+2g]. */
int pa_debug_download_grown(const pa_field *f, int lev, int box, int comp, double *host_grown);
/* Expanded FillBoundary descriptor table of a level: for every cell of every local grown FAB (nghost layers),
 * (src_box<<40 | linear index in the source box's valid region) or -1.  Same encoding as the oracle's. */
int pa_debug_fb_source_map(pa_hier *h, int lev, int nghost, int cross, int64_t *out, int64_t out_len);
/* Face flags of (lev, box, face): one uint16 per face-plane cell (t1 fastest): bits 0-1 = mask value at the ghost
 * cell (0 covered, 1 not_covered, 2 outside_domain), bits 2..9 = not_covered at tangential offsets
 * (-r,0) (+r,0) (0,-r) (0,+r) (-r,-r) (+r,-r) (-r,+r) (+r,+r).  Returns the number of cells (0 if the face
 * has no record, i.e. it is entirely covered by same-level boxes). */
int64_t pa_debug_face_flags(pa_hier *h, int lev, int box, int face, uint16_t *out, int64_t out_len);
/* Polynomial coefficients and order of the coarse-fine ghost formula of (lev, box, face). */
int pa_debug_face_coef(pa_hier *h, int lev, int box, int face, int *kind, int *nx, double coef[4]);

/* Neighbour links of (lev, GLOBAL box): per face (amrex::Orientation order) 5 ints: neighbour global box id or -1,
 * its owner rank, and rel[3] (neighbour-relative cell = own-relative cell + rel). */
int pa_debug_links(pa_hier *h, int lev, int box, int out[30]);

/* Multi-rank exchange plan, for parity of the plan itself: identity of the cell each send-slab slot carries /
 * each recv-slab slot expects, encoded (source level << 56 | global box << 32 | linear index in the box's valid
 * region).  which = 0: send slab, 1: recv slab.  Returns the slab length in cells (writes min(len, out_len)). */
int64_t pa_debug_exchange_ids(pa_hier *h, int which, int64_t *out, int64_t out_len);
/* The same for the exchange of pa_fill_patch(lev, nghost, interp_type) (pa_fill_patch_pack's send slab, the recv slab it
 * unpacks).  Returns a negative pa_status if the level is not properly nested for that ghost width. */
int64_t pa_debug_fill_patch_exchange_ids(pa_hier *h, int lev, int nghost, int interp_type, int which, int64_t *out, int64_t out_len);

/* Device self-test of the stencil kernels' branch-free IEEE sqrt / reciprocal / quotient forms (the flame normal's
 * nrm = -max(1e-14, sqrt(G.G)), n = G / nrm of Src/curvature.cpp:467-502) against the plain operators on n pseudo-random
 * operand sets covering every exponent of their ranges, zeros, denormals and overflow.  Returns the number of results
 * that differ in any bit (0 = identical), or -1 on error. */
int64_t pa_debug_selftest_math(int64_t n, uint64_t seed);
/* Which arithmetic the TMA stencil kernel uses for the flame normal: 0 = the branch-free forms, 1 = the plain IEEE
 * operators, -1 = not decided yet.  Decided once per process at the first flame-normal launch: PA_NORMAL_MATH=fast|plain
 * forces one; otherwise the library runs the self-test above on the device and keeps the branch-free forms only if not
 * one result bit differs (both forms compute the same IEEE results; the choice affects speed only). */
int pa_debug_normal_math(void);
/* Measured FP64 rate of the device for separate multiplies and adds (no FMA: the instruction mix bit parity with the
 * reference's CPU build imposes on pa_filter), in Gop/s: the roofline denominator of the filter for ghost widths >= 2. */
int pa_debug_fp64_rate(double *gops);
/* The multigrid preconditioner of pa_smooth on its own: with pa_smooth's inputs (o->smoothing_time > 0; o->precond, tol_rel
 * and max_iter are not used), runs ncycles steps of phi <- phi + B (c - A phi) from phi = c, B one V-cycle, and writes
 * max|c - A phi| / max|c| into resid[0 .. ncycles]: resid[0] before the first step, resid[n] after step n.  c goes into
 * out[comp_c], the last phi into out[comp_phi].
 * *nmg = the number of multigrid levels of level 0, level 0 itself included (1: level 0 does not coarsen). */
int pa_debug_smooth_vcycle(pa_field *state, int comp_S, double prog_min, double prog_max, const pa_smooth_opts *o, pa_field *out,
                           int comp_c, int comp_phi, int ncycles, double *resid, int *nmg);
/* 1 if curvature on this hierarchy runs through the fused kernel (every local box eligible: >= 3 cells in every direction,
 * <= 128 wide), 0 if it takes the separate flame-normal / divergence kernels, < 0 on error. */
int pa_debug_curv_fused(pa_hier *h);
/* kernels launched by the fused curvature path so far (fused kernel + shell pass), process-wide */
int64_t pa_debug_curv_fused_launches(void);

#ifdef __cplusplus
}
#endif
#endif
