// pa_types.h -- POD records shared by the host descriptor builder (hier.cpp) and the CUDA kernels.
// Every table is built once per hierarchy on the host, uploaded, and then reused by every ghost fill.
#ifndef PA_TYPES_H
#define PA_TYPES_H

#include <stdint.h>

#define PA_MAX_LEVELS 12
#define PA_MAX_BOX_SIDE 1024          // coarse gather index packs 3 x 10-bit box-relative coordinates

// valid region of a local box
struct PaBoxDev {
    int lo[3];
    int n[3];
};

// storage of one component of a local box inside the level slab (see DESIGN.md "data layout"):
// element (i,j,k) lives at off + (k-lo2+ng)*PS + (j-lo1+ng)*P + (i-lo0+ng+xoff)
struct PaLayDev {
    long long off;    // element offset inside one component's level slab
    int P;            // row pitch in doubles (a multiple of 4 by default: every row starts on a 32-byte sector; PA_ROW_ALIGN)
    int PS;           // plane stride = P * (ny + 2 ng)
    int xoff;         // lead pad so that the first VALID cell of each row is 32-byte aligned (at least 16: 128-bit accesses)
    int ng;
};

// same-level / periodic halo copy row == amrex CopyComTag {dbox, sbox, dstIndex, srcIndex}
// (AMReX_FabArrayBase.H:193-201): dst cell d in [dlo, dlo+n) of local box `dbox` <- src cell d+shift of `sbox`.
struct PaHaloTag {
    int dbox;         // local index of the receiving box
    int sbox;         // source box in the level's EXTENDED box index (local boxes first, then the peer-owned link
                      // targets, read through peer-mapped memory), or -1 if its data arrives in the recv slab
    int dlo[3];
    int n[3];
    int shift[3];
    int srank;        // rank that owns the source box
    long long start;  // first cell of this tag in the flattened cell enumeration of the table
    long long rsrc;   // sbox<0: first cell of this tag's data inside the recv slab (per component)
};

// Neighbour link of one (box, face): the whole width-1 ghost layer of the face lies inside ONE same-level box
// whose row pitch and plane stride equal this box's.  The stencil kernels then read the neighbour's valid cells
// in place (TMA bulk copies for y rows / z planes, scalar loads for x columns) and the ghost cells of that face
// are never materialised.  Neighbour-relative cell = own-relative cell + rel.
struct PaNbrFace {
    int nb;           // extended box index of the neighbour, -1 = face not linked (ghosts are materialised)
    int rank;         // owner of the neighbour (== own rank unless the hierarchy was created with peer links)
    int rel[3];
    int pad;
};
struct PaNbr {
    PaNbrFace f[6];   // amrex::Orientation order: low x,y,z, high x,y,z
};

// where rank r's slab of a (field, level) lives in this process' address space (own allocation or an IPC mapping)
struct PaPeerSlab {
    const double* base;   // component 0
    long long cs;         // component stride of that rank's slab
};

// what a rank must pack for a peer: src cells [slo, slo+n) of local box sbox -> send slab at soff
struct PaPackTag {
    int sbox;         // local source box
    int slev;         // level the source box belongs to
    int slo[3];
    int n[3];
    long long dense;  // prefix over cells in pack-table order (the kernel's enumeration)
    long long start;  // first cell of this tag inside the send slab
};

enum { PA_FACE_NEUMANN = 0, PA_FACE_REFLECT_ODD = 1, PA_FACE_CF = 2 };

// one record per (box, face) that has at least one ghost cell with mask > 0
struct PaFaceRec {
    int box;          // local box
    int face;         // 0..2 = low x,y,z ; 3..5 = high x,y,z  (amrex::Orientation order)
    int kind;         // PA_FACE_*
    int nx;           // NX = min(blen+1, maxorder=4)   (AMReX_MLLinOp_K.H:50)
    double coef[4];   // poly_interp_coeff(-0.5, {-bcl*dxinv, .5, 1.5, 2.5}, NX)
    int n1, n2;       // face-plane extent along the two tangential directions t1 < t2 (t1 fastest)
    int rlo1, rlo2;   // coarse register plane: low corner (coarse index space) along t1, t2
    int rn1, rn2;     // coarse register plane extent
    int ratio;        // refinement ratio to the coarse level
    int pad;
    long long start;  // first plane cell of this record in the flattened enumeration (= offset into flags[])
    long long cidx;   // first entry of this record's coarse gather index (rn1*rn2 entries), -1 if none
};

// coarse gather index entry: which coarse VALID cell a register cell reads
struct PaCrseIdx {
    int box;          // local coarse box, -1 = nothing copied there (reference leaves NaN), <= -2: remote slot -(box+2)
    unsigned rel;     // i | j<<10 | k<<20 relative to the coarse box's low corner (or remote slot offset)
};

// coarse gather OFFSET table (Hier::crse_offsets), one entry per register cell:
//   >= 0                       element offset inside this rank's coarse slab (one component)
//   -1                         nothing copied there (the reference leaves NaN)
//   -2 - slot                  slot of the recv slab (coarse cell of another rank, moved by the slab exchange)
//   -(PA_CRSE_PEER_BASE + (rank << PA_CRSE_PEER_SHIFT) + offset)   coarse cell of another rank, read in place through the
//                              peer mapping of that rank's slab (PA_HIER_PEER_LINKS)
#define PA_CRSE_PEER_BASE (1LL << 60)
#define PA_CRSE_PEER_SHIFT 44

// BC-fill work item: up to PA_FACE_CHUNK consecutive plane cells of one face record (one thread block each), so the
// kernel never searches for "which record does this cell belong to"
#define PA_FACE_CHUNK 128
struct PaFaceBlock {
    int rec;          // index into the face record table
    int cell0;        // first plane cell of the chunk, relative to the record's start
};

// a caller's device array (pa_array4) resolved against one local box: cell (i,j,k) relative to the box's low corner,
// component m of the copied range, lives at p[i + j*js + k*ks + m*ns]
struct PaA4Dev {
    double* p;
    long long js, ks, ns;
};
// device <-> field copy work item (pa_field_upload_device): rows [row0, row0+nrows) of local box `box`, row = k*ny + j
struct PaRowItem {
    int box;
    int row0, nrows;
    int pad;
};

// stencil work item: rows [y0, y0+ny) x planes [z0, z0+nz) of a local box, full x extent
struct PaTile {
    int lev;
    int box;
    int y0, ny;
    int z0, nz;
};

// ---- FillPatchTwoLevels bookkeeping of the filterPlt path (FabArrayBase::FPinfo, AMReX_FabArrayBase.cpp) --------------
// A "piece" is a box of ghost cells of one fine box that lie inside the domain and that no fine box covers: they are
// interpolated from the next coarser level.  Its coarse patch = coarsen(piece, ratio) grown by the interpolater's stencil
// (1 cell for the conservative linear one, 0 for piecewise constant) lives in a scratch buffer, gathered from the coarse
// level's VALID cells; coarse patch cells outside the domain are never stored -- readers clamp the index (first-order
// extrapolation, AMReX_FilCC_3D_C.H).
struct PaFpPiece {
    int box;            // local fine box the ghost cells belong to
    int lo[3], n[3];    // the piece (fine index space)
    int clo[3], cn[3];  // coarse patch box (coarse index space), may stick out of the coarse domain
    long long cstart;   // first cell of the coarse patch in the scratch buffer (per component)
    long long fstart;   // prefix over the fine cells of all pieces (the interpolation kernel's enumeration)
};
// coarse VALID cells [lo, lo+n) of local coarse box sbox -> coarse patch of piece `piece`
struct PaFpCopy {
    int piece;
    int sbox;
    int lo[3], n[3];
    long long start;    // prefix over the cells of all copy tags
};
// several ranks: recv-slab cells [rsrc, rsrc + n) -> cells [lo, lo+n) of a ghost region of a local box (same-level source
// owned by another rank, box >= 0) or of the coarse patch of piece -1 - box (coarse source owned by another rank)
struct PaFpUnpack {
    int box;            // >= 0: local fine box (fine index space); < 0: piece -1 - box (coarse index space)
    int lo[3], n[3];
    int pad;
    long long rsrc;     // first cell of this record inside the recv slab (per component)
    long long start;    // prefix over the cells of all unpack records (the kernel's enumeration)
};
// a local box whose grown region leaves the domain: its ghost cells outside take the value at the clamped index
struct PaFpClamp {
    int box;
    int pad;
    long long start;    // prefix over the cells of the grown boxes in this list
};

// ---- composite implicit-diffusion solve (pa_smooth, smooth.cu) ----------------------------------------------------------
// coarse cells [lo, lo+n) (coarse index space) of local coarse box cbox are covered by local fine box fbox: they hold the
// average of their 8 fine cells (average_down)
struct PaAvgDown {
    int cbox, fbox;
    int lo[3], n[3];
    long long start;    // prefix over the cells of all records of the coarse level (the kernel's enumeration)
};
// one coarse-fine face seen from the coarse side: the face `side` (0 low, 1 high) along `dir` of the uncovered coarse cell c
// (box-relative in local coarse box cbox) borders the fine region; its flux is replaced by the average of the 4 fine face
// fluxes between the fine cells f + (0 | 1 along the two tangential directions) (box-relative in local fine box fbox, the
// first fine cells inside the fine region) and their coarse-fine ghost cells
struct PaReflux {
    int cbox, fbox;
    int c[3], f[3];
    int dir, side;
};

// face flags (uint16 per face-plane cell)
#define PA_FLAG_MASK(f)   ((f) & 3)
#define PA_FLAG_NC(f, b)  (((f) >> (2 + (b))) & 1)   // b: 0 (-r,0) 1 (+r,0) 2 (0,-r) 3 (0,+r) 4 (-,-) 5 (+,-) 6 (-,+) 7 (+,+)

#endif
