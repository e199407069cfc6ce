// hier.hpp -- host-side AMR hierarchy metadata and copy-descriptor tables (no CUDA in this file).
#ifndef PA_HIER_HPP
#define PA_HIER_HPP

#include <array>
#include <cstdint>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "pa_types.h"

namespace pa {

struct Box {
    int lo[3], hi[3];
    bool ok() const { return lo[0] <= hi[0] && lo[1] <= hi[1] && lo[2] <= hi[2]; }
    int len(int d) const { return hi[d] - lo[d] + 1; }
    long long npts() const { return (long long)len(0) * len(1) * len(2); }
    bool contains(int i, int j, int k) const {
        return i >= lo[0] && i <= hi[0] && j >= lo[1] && j <= hi[1] && k >= lo[2] && k <= hi[2];
    }
    Box grown(int n) const { Box b = *this; for (int d = 0; d < 3; ++d) { b.lo[d] -= n; b.hi[d] += n; } return b; }
    Box shifted(const int* s) const { Box b = *this; for (int d = 0; d < 3; ++d) { b.lo[d] += s[d]; b.hi[d] += s[d]; } return b; }
    Box isect(const Box& o) const {
        Box b = *this;
        for (int d = 0; d < 3; ++d) { if (o.lo[d] > b.lo[d]) b.lo[d] = o.lo[d]; if (o.hi[d] < b.hi[d]) b.hi[d] = o.hi[d]; }
        return b;
    }
};

inline int coarsen(int i, int r) { return (i < 0) ? -((-i + r - 1) / r) : i / r; }

// Uniform-bin hash of a level's boxes for intersection queries (the role of BoxArray::intersections).
class BoxHash {
public:
    void build(const std::vector<Box>& boxes);
    // calls fn(box_index, intersection) for every box meeting q
    template <class F> void query(const Box& q, F&& fn) const;
private:
    const std::vector<Box>* boxes_ = nullptr;
    int bin_[3] = {1, 1, 1};
    int maxlen_[3] = {1, 1, 1};
    std::unordered_map<uint64_t, std::vector<int>> bins_;
    static uint64_t key(int a, int b, int c) {
        return ((uint64_t)(uint32_t)(a + (1 << 20)) << 42) | ((uint64_t)(uint32_t)(b + (1 << 20)) << 21) | (uint64_t)(uint32_t)(c + (1 << 20));
    }
    static int fdiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
};

template <class F>
void BoxHash::query(const Box& q, F&& fn) const {
    int blo[3], bhi[3];
    for (int d = 0; d < 3; ++d) {
        blo[d] = fdiv(q.lo[d] - maxlen_[d] + 1, bin_[d]);
        bhi[d] = fdiv(q.hi[d], bin_[d]);
    }
    for (int c = blo[2]; c <= bhi[2]; ++c)
        for (int b = blo[1]; b <= bhi[1]; ++b)
            for (int a = blo[0]; a <= bhi[0]; ++a) {
                auto it = bins_.find(key(a, b, c));
                if (it == bins_.end()) continue;
                for (int idx : it->second) {
                    Box is = q.isect((*boxes_)[idx]);
                    if (is.ok()) fn(idx, is);
                }
            }
}

struct Level {
    Box dom;
    double dx[3], dxinv[3];
    int ratio = 1;                    // to the next coarser level
    std::vector<Box> boxes;           // global BoxArray
    std::vector<int> owner;           // global DistributionMapping
    std::vector<int> local;           // global ids of this rank's boxes, ascending
    std::vector<int> g2l;             // global id -> local index or -1
    // extended box index: this rank's boxes first (same order as `local`), then the boxes of other ranks that are
    // neighbour-link targets of local boxes (read in place through peer-mapped memory)
    std::vector<int> ext;             // extended index -> global id
    std::vector<int> g2e;             // global id -> extended index or -1
    // neighbour links of EVERY box of the level (global id x 6 faces): sender and receiver must agree on them
    struct Link { int nb = -1; int shift[3] = {0, 0, 0}; };
    std::vector<std::array<Link, 6>> link;
    std::vector<PaNbr> nbr;           // device form, per local box
    BoxHash hash;
    long long ncells = 0, ncells_local = 0;
};

// Layout of one component of every local box of a level for a given ghost width.
struct Layout {
    int ng = 0;
    std::vector<PaLayDev> lay;        // per box of the extended index (peer boxes: offsets inside THEIR rank's slab)
    std::vector<PaLayDev> all;        // per GLOBAL box id: the box's place inside its owner's slab
    long long comp_stride = 0;        // elements per component of this rank's level slab (multiple of 16)
    std::vector<long long> rank_comp_stride;   // the same for every rank
};

// Everything the ghost-fill kernels need for one level at one "mode".
struct HaloTable {
    // order: [faces without a neighbour link: local sources, then recv-slab sources][linked faces]
    // The product path copies only the first group (the stencil reads linked faces in place); pa_fill_ghosts /
    // pa_fill_boundary materialise both.
    std::vector<PaHaloTag> tags;
    long long ncells = 0;             // total cells over all tags
    int nlocal_tags = 0;
    int ntags_unlinked = 0;
    long long ncells_unlinked = 0;
};

struct FaceTable {                    // all levels concatenated, level-major
    std::vector<PaFaceRec> recs;
    std::vector<int> rec_level;       // level of each record
    std::vector<uint16_t> flags;
    std::vector<PaCrseIdx> cidx;
    std::vector<long long> level_rec_begin;   // nlev+1
    std::vector<PaFaceBlock> blocks;          // chunks of <= PA_FACE_CHUNK plane cells, record-major (hence level-major)
    std::vector<long long> level_blk_begin;   // nlev+1
    long long ncells = 0;
};

// Per-peer exchange plan for one exchange step covering levels [0,nlev): what this rank receives from / packs for
// every peer.  Cell counts are per component.
struct ExchangePlan {
    std::vector<PaPackTag> pack;                      // canonical order: fill level, dst box, ...
    std::vector<long long> pack_level_begin;          // nlev+1: first pack tag of each FILL level
    std::vector<long long> send_prefix;               // nranks+1, in cells
    std::vector<long long> recv_prefix;               // nranks+1, in cells
    std::vector<std::vector<long long>> level_send_cell0;  // [level][peer]: first send-slab cell of the level's block for the peer (nlev+1 rows)
    std::vector<std::vector<long long>> level_recv_cell0;  // [level][peer]: same on the receive side
    // debug / parity: global identity (src level<<56 | global box<<32 | linear index in its valid region) of the cell every
    // recv-slab slot expects, and of the cell every send-slab slot carries
    std::vector<long long> recv_ids, send_ids;
};

// Ghost-cell fill of the filterPlt path for one (level, ghost width, interpolater stencil width): see PaFpPiece.
struct FillPatchTable {
    std::vector<PaFpPiece> pieces;
    std::vector<PaFpCopy> copies;
    std::vector<PaFpClamp> clamps;
    long long nfine = 0;              // fine cells to interpolate
    long long ncrse = 0;              // scratch cells (per component)
    long long ncopy = 0;              // coarse cells gathered
    long long nclamp = 0;             // cells of the grown boxes in `clamps`
    std::string err;                  // non-empty: the coarse level does not cover a coarse patch (improper nesting); decided
                                      // over every box of the level, so all ranks reach the same verdict
    // Several ranks: the sources owned by another rank than the destination box's, moved as packed slabs ([cell][comp]).
    // Every rank walks every box of the level in global id order (same-level sources, then coarse copies piece by piece);
    // the stream from rank p to rank q is the subsequence with source owner p and destination owner q, so both sides agree
    // on slab offsets without a handshake.  Empty on one rank.
    std::vector<PaPackTag> pack;      // what this rank packs (slev = l: same-level source, l - 1: coarse source)
    std::vector<PaFpUnpack> unpack;   // recv-slab cells -> ghost cells / coarse-patch cells of this rank
    std::vector<long long> send_prefix, recv_prefix;   // nranks+1, in cells
    long long npack = 0, nunpack = 0; // cells
    // debug / parity: identity of the cell every send-slab slot carries / recv-slab slot expects (ExchangePlan's form)
    std::vector<long long> send_ids, recv_ids;
};

// Tables of the composite implicit-diffusion solve (pa_smooth), built on its first call on a hierarchy.
struct SmoothTables {
    std::string err;                          // non-empty: the hierarchy is not supported (message says why)
    std::vector<PaFaceRec> recs;              // faces.recs with the smoothing operator's coarse-fine polynomial order
    std::vector<PaAvgDown> avg;               // level-major by COARSE level
    std::vector<long long> avg_begin;         // nlev+1: first record of each coarse level
    std::vector<long long> avg_cells;         // nlev: covered cells of each coarse level
    std::vector<PaReflux> reflux;             // sorted by (coarse level, dir, side)
    std::vector<long long> reflux_begin;      // nlev*6+1: first record of each (coarse level, 2*dir+side)
    // multigrid preconditioner: level 0 and its coarsenings by 2 (MG level k+1 = MG level k with every box and the domain
    // coarsened; it exists while every box of level k is coarsenable -- even low corner and length -- and the coarsened length is
    // at least 2).  mg_boxes[0] / mg_dom[0] are level 0 itself; box b of MG level k+1 is box b of level k coarsened.
    std::vector<std::vector<Box>> mg_boxes;
    std::vector<Box> mg_dom;
    std::vector<PaAvgDown> mg_avg;            // restriction / prolongation between MG levels k and k+1: one record per box
    std::vector<long long> mg_avg_begin;      // nmg: first record of each (k, k+1) pair; [nmg-1] = end
    std::vector<long long> mg_avg_cells;      // nmg-1: cells of MG level k+1
};

// BoxList::maxSize: every box replaced, in place, by its chunks no longer than max_grid_size (AMReX_BoxList.cpp:765-815)
void box_max_size(int nboxes, const int* boxes, int max_grid_size, std::vector<Box>& out);

class Hier {
public:
    int nlev = 0;
    int rank = 0, nranks = 1;
    bool peer_links = false;          // links may cross ranks (every rank's slabs are peer-mapped, PA_HIER_PEER_LINKS)
    bool no_links = false;            // PA_HIER_NO_LINKS: materialise every ghost cell (reference-style data flow)
    bool filter_only = false;         // PA_HIER_FILTER_ONLY: grids of the filterPlt path (no ratio alignment, no face tables)
    int is_per[3] = {1, 1, 1};
    int bc_kind[3] = {0, 0, 0};
    std::vector<Level> lev;
    double build_seconds = 0.0;

    // descriptor tables (cross / width-1 mode used by the product path)
    std::vector<HaloTable> halo_cross;        // per level
    FaceTable faces;
    ExchangePlan xplan;

    std::string init(int nlev, const struct pa_level_desc_host* L, const int* is_per, const int* bc_kind, int rank, int nranks,
                     unsigned flags = 0);
    bool linked(int l, int gb, int face) const { return lev[l].link[gb][face].nb >= 0; }

    const Layout& layout(int l, int ng);      // lazily built, cached
    // coarse gather index resolved against the ng-ghost layout: element offset inside the coarse level's component slab,
    // -1 = never filled (NaN in the reference), <= -2: recv-slab slot -(v+2)
    std::vector<long long> crse_offsets(int ng);
    // full FillBoundary table (all ng layers incl. edges/corners) -- debug / pa_fill_boundary(cross=0); sources owned by
    // this rank only (on several ranks the others arrive through fill_patch's exchange)
    const HaloTable& halo_full(int l, int ng);
    // FillPatchTwoLevels / FillPatchSingleLevel tables of level l for ng ghost layers; cgrow = coarse cells the
    // interpolater reads around the coarsened piece, with the exchange plan of the cross-rank sources.  Non-periodic only.
    const FillPatchTable& fill_patch(int l, int ng, int cgrow);
    // covered-cell, reflux and coarse-fine coefficient tables of pa_smooth (lazily built, cached; one rank, ratio 2)
    const SmoothTables& smooth_tables(int maxorder);

    void periodic_shifts(const Box& dom, int ng, std::vector<std::array<int, 3>>& out) const;

private:
    std::map<std::pair<int, int>, Layout> layouts_;
    std::map<std::pair<int, int>, HaloTable> halo_full_;
    std::map<std::array<int, 3>, FillPatchTable> fill_patch_;
    std::map<int, SmoothTables> smooth_;
    void build_links();
    void build_halo(int l, int ng, bool cross, HaloTable& out, bool allow_remote);
    std::string build_faces();
    void build_exchange();
};

struct pa_level_desc_host {
    int domain_lo[3], domain_hi[3];
    double dx[3];
    int nboxes;
    const int* boxes;
    const int* owner;
};

void sfc_distribute(int nboxes, const int* boxes, int nranks, int* owner_out);

}  // namespace pa
#endif
