// hier.cpp -- builds, on the host, the integer descriptor tables of the ghost fill:
//   * same-level / periodic halo rows            (what FabArrayBase::FB caches, AMReX_FabArrayBase.cpp:658-877)
//   * face masks, compressed to per-cell flags   (MultiMask::define, AMReX_MultiMask.cpp:25-71; the two mask sets of
//                                                 MLCellLinOp::defineAuxData and BndryData::define)
//   * box-face boundary records + coefficients   (MLMGBndry::setBoxBC, AMReX_MLMGBndry.H:107-155; AMReX_MLLinOp_K.H:48-53)
//   * coarse gather index of every c-f face      (BndryRegister on the coarsened box + copyFrom of coarse valid cells,
//                                                 AMReX_BndryRegister.H:147-190,266-276)
//   * the per-peer exchange plan when boxes are spread over several ranks (one process per GPU)
// Integer work only; the arithmetic it mirrors is box algebra, so results are index-exact by construction
// and are checked cell by cell against the oracle in tests/.
#include "hier.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace pa {

void BoxHash::build(const std::vector<Box>& boxes) {
    boxes_ = &boxes;
    bins_.clear();
    for (int d = 0; d < 3; ++d) maxlen_[d] = 1;
    for (const Box& b : boxes)
        for (int d = 0; d < 3; ++d) maxlen_[d] = std::max(maxlen_[d], b.len(d));
    for (int d = 0; d < 3; ++d) bin_[d] = maxlen_[d];
    for (size_t i = 0; i < boxes.size(); ++i) {
        const Box& b = boxes[i];
        bins_[key(fdiv(b.lo[0], bin_[0]), fdiv(b.lo[1], bin_[1]), fdiv(b.lo[2], bin_[2]))].push_back((int)i);
    }
}

// Periodicity::shiftIntVect (AMReX_Periodicity.cpp:8-33)
void Hier::periodic_shifts(const Box& dom, int ng, std::vector<std::array<int, 3>>& out) const {
    int per[3] = {0, 0, 0}, jmp[3] = {1, 1, 1};
    for (int d = 0; d < 3; ++d)
        if (is_per[d]) {
            int period = dom.len(d);
            per[d] = jmp[d] = period;
            while (per[d] < ng) per[d] += period;
        }
    out.clear();
    for (int i = -per[0]; i <= per[0]; i += jmp[0])
        for (int j = -per[1]; j <= per[1]; j += jmp[1])
            for (int k = -per[2]; k <= per[2]; k += jmp[2]) out.push_back({i, j, k});
}

static Box face_plane(const Box& b, int face, int out_layer /*1 = adjacent ghost layer*/, int extent) {
    int d = face % 3;
    Box r = b;
    for (int t = 0; t < 3; ++t)
        if (t != d) { r.lo[t] -= extent; r.hi[t] += extent; }
    if (face < 3) r.lo[d] = r.hi[d] = b.lo[d] - out_layer;
    else r.lo[d] = r.hi[d] = b.hi[d] + out_layer;
    return r;
}

// box minus box -> up to 6 disjoint boxes (amrex::boxDiff)
static void box_diff(const Box& a, const Box& b, std::vector<Box>& out) {
    Box is = a.isect(b);
    if (!is.ok()) { out.push_back(a); return; }
    Box rem = a;
    for (int d = 0; d < 3; ++d) {
        if (rem.lo[d] < is.lo[d]) { Box p = rem; p.hi[d] = is.lo[d] - 1; out.push_back(p); rem.lo[d] = is.lo[d]; }
        if (rem.hi[d] > is.hi[d]) { Box p = rem; p.lo[d] = is.hi[d] + 1; out.push_back(p); rem.hi[d] = is.hi[d]; }
    }
}

std::string Hier::init(int nlev_, const pa_level_desc_host* L, const int* per, const int* bck, int rank_, int nranks_,
                       unsigned flags) {
    auto t0 = std::chrono::steady_clock::now();
    peer_links = (flags & 1u) != 0;
    no_links = (flags & 2u) != 0;
    filter_only = (flags & 4u) != 0;
    if (nlev_ < 1 || nlev_ > PA_MAX_LEVELS) return "number of levels must be in [1," + std::to_string(PA_MAX_LEVELS) + "]";
    if (nranks_ < 1 || rank_ < 0 || rank_ >= nranks_) return "bad rank / nranks";
    nlev = nlev_; rank = rank_; nranks = nranks_;
    for (int d = 0; d < 3; ++d) { is_per[d] = per[d] ? 1 : 0; bc_kind[d] = bck ? bck[d] : 0; }
    lev.assign(nlev, Level());
    for (int l = 0; l < nlev; ++l) {
        Level& V = lev[l];
        for (int d = 0; d < 3; ++d) {
            V.dom.lo[d] = L[l].domain_lo[d]; V.dom.hi[d] = L[l].domain_hi[d];
            V.dx[d] = L[l].dx[d];
            if (!(V.dx[d] > 0.0)) return "dx must be positive";
            V.dxinv[d] = 1.0 / V.dx[d];                       // Geometry: inv_dx = 1/dx (AMReX_Geometry.cpp:521)
        }
        if (!V.dom.ok()) return "empty domain on level " + std::to_string(l);
        if (l > 0) {
            // ratio from the level domains (AMReX_MLLinOp.H:856-885)
            int r = V.dom.len(0) / lev[l - 1].dom.len(0);
            for (int d = 0; d < 3; ++d)
                if (lev[l - 1].dom.len(d) * r != V.dom.len(d) || V.dom.lo[d] != lev[l - 1].dom.lo[d] * r)
                    return "level " + std::to_string(l) + " domain is not an isotropic refinement of the coarser domain";
            if (r != 2 && r != 4) return "refinement ratio must be 2 or 4 (got " + std::to_string(r) + ")";
            V.ratio = r;
        }
        if (L[l].nboxes < 1) return "level " + std::to_string(l) + " has no boxes";
        V.boxes.resize(L[l].nboxes); V.owner.resize(L[l].nboxes); V.g2l.assign(L[l].nboxes, -1);
        for (int b = 0; b < L[l].nboxes; ++b) {
            Box& B = V.boxes[b];
            for (int d = 0; d < 3; ++d) { B.lo[d] = L[l].boxes[6 * b + d]; B.hi[d] = L[l].boxes[6 * b + 3 + d]; }
            if (!B.ok()) return "empty box";
            for (int d = 0; d < 3; ++d) {
                if (B.lo[d] < V.dom.lo[d] || B.hi[d] > V.dom.hi[d]) return "box outside its level domain";
                if (B.len(d) > PA_MAX_BOX_SIDE) return "box side > " + std::to_string(PA_MAX_BOX_SIDE) + " cells is not supported";
                if (l > 0 && !filter_only && (coarsen(B.lo[d], V.ratio) * V.ratio != B.lo[d] || (B.hi[d] + 1) % V.ratio != 0))
                    return "fine box is not aligned to the refinement ratio";
            }
            int o = L[l].owner ? L[l].owner[b] : 0;
            if (o < 0 || o >= nranks) return "box owner out of range";
            V.owner[b] = o;
            V.ncells += B.npts();
            if (o == rank) { V.g2l[b] = (int)V.local.size(); V.local.push_back(b); V.ncells_local += B.npts(); }
        }
        V.hash.build(V.boxes);
    }
    build_links();
    halo_cross.assign(nlev, HaloTable());
    xplan = ExchangePlan();
    xplan.send_prefix.assign(nranks + 1, 0);
    xplan.recv_prefix.assign(nranks + 1, 0);
    xplan.pack_level_begin.assign(nlev + 1, 0);
    // a filter-only hierarchy on several ranks moves its cross-rank cells through fill_patch's own plan: the width-1 cross
    // tables (and the ratio-aligned coarse needs they assume) would never be used
    const bool cross_tables = !(filter_only && nranks > 1);
    if (nranks > 1 && cross_tables) build_exchange();          // fixes recv/send slab offsets first
    if (cross_tables)
        for (int l = 0; l < nlev; ++l) build_halo(l, 1, true, halo_cross[l], true);
    if (filter_only) {                             // FillPatch needs no face masks / BC records; grids may be unaligned
        faces = FaceTable();
        faces.level_rec_begin.assign(nlev + 1, 0);
        faces.level_blk_begin.assign(nlev + 1, 0);
    } else {
        std::string e = build_faces();
        if (!e.empty()) return e;
    }
    build_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return "";
}

static int row_align_doubles() {
    static const int v = [] {
        const char* e = getenv("PA_ROW_ALIGN");
        const int b = e ? atoi(e) : 32;
        return (b == 16 || b == 32 || b == 64 || b == 128) ? b / 8 : 4;
    }();
    return v;
}

const Layout& Hier::layout(int l, int ng) {
    auto key = std::make_pair(l, ng);
    auto it = layouts_.find(key);
    if (it != layouts_.end()) return it->second;
    Layout Y;
    Y.ng = ng;
    const Level& V = lev[l];
    // every rank packs ITS boxes (ascending global id) back to back, so any rank can compute any other rank's layout
    std::vector<PaLayDev> all(V.boxes.size());
    Y.rank_comp_stride.assign(nranks, 0);
    for (size_t gb = 0; gb < V.boxes.size(); ++gb) {
        const Box& B = V.boxes[gb];
        long long& off = Y.rank_comp_stride[V.owner[gb]];
        PaLayDev e;
        e.ng = ng;
        // The first valid cell of every row is aligned to `ra` doubles and the pitch is a multiple of it.  ra = 4 (32 bytes, one
        // DRAM / L2 sector): with 16-byte alignment a full-row store of a field with one ghost cell wrote HALF of its first and
        // last sector, and ncu counted 25 M partial-sector (ECC read-modify-write) operations and 0.8 GB of extra DRAM reads per
        // flame-normal pass -- two per row and component -- against 62 for the gradient kernel, whose output field has no ghost
        // cells (profiles/r02_ablate_normal_f3.txt).  PA_ROW_ALIGN=16|32|64|128 (bytes) overrides.
        const int ra = row_align_doubles();
        e.xoff = (ra - ng % ra) % ra;
        int w = e.xoff + B.len(0) + 2 * ng;
        e.P = (w + ra - 1) / ra * ra;
        e.PS = e.P * (B.len(1) + 2 * ng);
        e.off = off;
        long long sz = (long long)e.PS * (B.len(2) + 2 * ng);
        off += (sz + 15) & ~15LL;                          // every box starts 128-byte aligned
        all[gb] = e;
    }
    for (int gb : V.ext) Y.lay.push_back(all[gb]);
    Y.all = all;
    Y.comp_stride = Y.rank_comp_stride[rank];
    return layouts_.emplace(key, std::move(Y)).first->second;
}

// ---------------------------------------------------------------------------------------------------------
// Canonical enumeration of everything a destination box needs from other boxes for a width-1 cross ghost fill.
// Both the receiver (building its tables) and the sender (building its pack list) walk this in the same order.
// ---------------------------------------------------------------------------------------------------------
namespace {
struct HaloNeed { int face; int sbox; Box dst; int shift[3]; };        // dst region (dst index space), src = dst+shift in sbox
struct CrseNeed { int face; int cbox; Box reg; int shift[3]; };        // register cells `reg` (coarse idx space) <- cbox cells reg+shift
}

static void sort_isects(std::vector<std::pair<int, Box>>& v) {
    std::sort(v.begin(), v.end(), [](const std::pair<int, Box>& a, const std::pair<int, Box>& b) { return a.first < b.first; });
}

enum { NEED_ALL = 0, NEED_UNLINKED = 1, NEED_LINKED = 2 };

static void halo_needs_cross(const Hier& H, int l, int gb, std::vector<HaloNeed>& out, int which = NEED_ALL) {
    const Level& V = H.lev[l];
    std::vector<std::array<int, 3>> sh;
    H.periodic_shifts(V.dom, 1, sh);
    std::vector<std::pair<int, Box>> is;
    for (int face = 0; face < 6; ++face) {
        if (which != NEED_ALL && H.linked(l, gb, face) != (which == NEED_LINKED)) continue;
        Box slab = face_plane(V.boxes[gb], face, 1, 0);
        for (auto& s : sh) {
            is.clear();
            V.hash.query(slab.shifted(s.data()), [&](int k, const Box& ib) { is.emplace_back(k, ib); });
            sort_isects(is);
            for (auto& e : is) {
                HaloNeed n;
                n.face = face; n.sbox = e.first;
                int neg[3] = {-s[0], -s[1], -s[2]};
                n.dst = e.second.shifted(neg);
                for (int d = 0; d < 3; ++d) n.shift[d] = s[d];
                out.push_back(n);
            }
        }
    }
}

static Box crse_register_box(const Box& fine, int ratio, int face) {
    Box cb;
    for (int d = 0; d < 3; ++d) { cb.lo[d] = coarsen(fine.lo[d], ratio); cb.hi[d] = coarsen(fine.hi[d], ratio); }
    return face_plane(cb, face, 1, 2);              // in 0, out 1, extent 2 (AMReX_MLCellLinOp.H:461-469)
}

static void crse_needs(const Hier& H, int l, int gb, int face, std::vector<CrseNeed>& out) {
    const Level& V = H.lev[l];
    const Level& C = H.lev[l - 1];
    Box rb = crse_register_box(V.boxes[gb], V.ratio, face);
    std::vector<std::array<int, 3>> sh;
    H.periodic_shifts(C.dom, 0, sh);
    std::vector<std::pair<int, Box>> is;
    for (auto& s : sh) {
        is.clear();
        C.hash.query(rb.shifted(s.data()), [&](int k, const Box& ib) { is.emplace_back(k, ib); });
        sort_isects(is);
        for (auto& e : is) {
            CrseNeed n;
            n.face = face; n.cbox = e.first;
            int neg[3] = {-s[0], -s[1], -s[2]};
            n.reg = e.second.shifted(neg);
            for (int d = 0; d < 3; ++d) n.shift[d] = s[d];
            out.push_back(n);
        }
    }
}

// mask of a face plane grown tangentially by `extent`: 0 covered, 1 not_covered, 2 outside_domain
static void plane_mask(const Hier& H, int l, const Box& plane, int grow_domain, std::vector<uint8_t>& m) {
    const Level& V = H.lev[l];
    Box dom = V.dom;
    for (int d = 0; d < 3; ++d)
        if (H.is_per[d]) { dom.lo[d] -= grow_domain; dom.hi[d] += grow_domain; }
    int n0 = plane.len(0), n1 = plane.len(1);
    m.assign((size_t)plane.npts(), 0);
    for (int k = plane.lo[2]; k <= plane.hi[2]; ++k)
        for (int j = plane.lo[1]; j <= plane.hi[1]; ++j)
            for (int i = plane.lo[0]; i <= plane.hi[0]; ++i)
                m[((size_t)(k - plane.lo[2]) * n1 + (j - plane.lo[1])) * n0 + (i - plane.lo[0])] = dom.contains(i, j, k) ? 1 : 2;
    std::vector<std::array<int, 3>> sh;
    H.periodic_shifts(V.dom, 0, sh);
    for (auto& s : sh)
        V.hash.query(plane.shifted(s.data()), [&](int, const Box& ib) {
            for (int k = ib.lo[2]; k <= ib.hi[2]; ++k)
                for (int j = ib.lo[1]; j <= ib.hi[1]; ++j)
                    for (int i = ib.lo[0]; i <= ib.hi[0]; ++i)
                        m[((size_t)(k - s[2] - plane.lo[2]) * n1 + (j - s[1] - plane.lo[1])) * n0 + (i - s[0] - plane.lo[0])] = 0;
        });
}

// Does (level, box, face) carry a boundary record, i.e. is any adjacent ghost cell not covered by a same-level box?
// Cheap pre-test shared by the receiver and the sender so that both enumerate the same coarse needs.
static bool face_has_uncovered(const Hier& H, int l, int gb, int face) {
    const Level& V = H.lev[l];
    Box plane = face_plane(V.boxes[gb], face, 1, 0);
    long long covered = 0;
    std::vector<std::array<int, 3>> sh;
    H.periodic_shifts(V.dom, 0, sh);
    for (auto& s : sh)
        V.hash.query(plane.shifted(s.data()), [&](int, const Box& ib) { covered += ib.npts(); });
    return covered < plane.npts();       // valid boxes are disjoint, so the covered pieces never overlap
}

static bool face_is_physical(const Hier& H, int l, int gb, int face) {
    const Level& V = H.lev[l];
    int d = face % 3;
    bool at = (face < 3) ? (V.boxes[gb].lo[d] == V.dom.lo[d]) : (V.boxes[gb].hi[d] == V.dom.hi[d]);
    return at && !H.is_per[d];
}

static inline long long cell_id(int lev, int gbox, const Box& B, int i, int j, int k) {
    long long lin = ((long long)(k - B.lo[2]) * B.len(1) + (j - B.lo[1])) * B.len(0) + (i - B.lo[0]);
    return ((long long)lev << 56) | ((long long)gbox << 32) | lin;
}

// Neighbour links (see PaNbrFace): face `f` of box gb is linked when its width-1 ghost layer, under exactly one
// periodic shift, lies inside exactly one same-level box with the same x and y extent (=> same row pitch and plane
// stride, so "ghost address + constant" addresses the neighbour's cell), owned by the same rank unless peer links
// are enabled.  Computed for every box of the level because senders must know which of a peer's faces are linked.
void Hier::build_links() {
    for (int l = 0; l < nlev; ++l) {
        Level& V = lev[l];
        V.link.assign(V.boxes.size(), std::array<Level::Link, 6>());
        V.ext = V.local;
        V.g2e.assign(V.boxes.size(), -1);
        for (size_t lb = 0; lb < V.local.size(); ++lb) V.g2e[V.local[lb]] = (int)lb;
        if (no_links) { V.nbr.assign(V.local.size(), PaNbr()); for (auto& n : V.nbr) for (auto& f : n.f) { f.nb = -1; f.rank = rank; f.rel[0] = f.rel[1] = f.rel[2] = 0; f.pad = 0; } continue; }
        std::vector<std::array<int, 3>> sh;
        periodic_shifts(V.dom, 1, sh);
        for (int gb = 0; gb < (int)V.boxes.size(); ++gb) {
            const Box& B = V.boxes[gb];
            for (int face = 0; face < 6; ++face) {
                Box plane = face_plane(B, face, 1, 0);
                int hits = 0, hk = -1;
                std::array<int, 3> hs{0, 0, 0};
                long long hn = 0;
                for (auto& s : sh)
                    V.hash.query(plane.shifted(s.data()), [&](int k, const Box& ib) { ++hits; hk = k; hs = s; hn = ib.npts(); });
                if (hits != 1 || hn != plane.npts()) continue;
                const Box& N = V.boxes[hk];
                if (N.len(0) != B.len(0) || N.len(1) != B.len(1)) continue;
                if (face % 3 == 0 && B.len(0) < 3) continue;        // the x-pair kernels want distinct first / last pairs
                if (V.owner[hk] != V.owner[gb] && !peer_links) continue;
                Level::Link& K = V.link[gb][face];
                K.nb = hk;
                for (int d = 0; d < 3; ++d) K.shift[d] = hs[d];
            }
        }
        // extended index: peer-owned link targets of local boxes
        for (int gb : V.local)
            for (int face = 0; face < 6; ++face) {
                int k = V.link[gb][face].nb;
                if (k >= 0 && V.g2e[k] < 0) { V.g2e[k] = (int)V.ext.size(); V.ext.push_back(k); }
            }
        V.nbr.assign(V.local.size(), PaNbr());
        for (size_t lb = 0; lb < V.local.size(); ++lb) {
            const Box& B = V.boxes[V.local[lb]];
            for (int face = 0; face < 6; ++face) {
                const Level::Link& K = V.link[V.local[lb]][face];
                PaNbrFace& F = V.nbr[lb].f[face];
                F.nb = (K.nb >= 0) ? V.g2e[K.nb] : -1;
                F.rank = (K.nb >= 0) ? V.owner[K.nb] : rank;
                for (int d = 0; d < 3; ++d) F.rel[d] = (K.nb >= 0) ? B.lo[d] + K.shift[d] - V.boxes[K.nb].lo[d] : 0;
                F.pad = 0;
            }
        }
    }
}

void Hier::build_exchange() {
    // Walk every (level, dst box) in canonical order; entries whose source owner differs from the dst owner are
    // exchanged.  The stream from rank p to rank q is the subsequence with (src owner p, dst owner q); both sides
    // enumerate it identically, so slab offsets agree without any handshake.
    struct Ent { int lev; int peer; PaPackTag t; };
    std::vector<Ent> sends;
    std::vector<std::vector<long long>> send_lvl(nlev, std::vector<long long>(nranks, 0)), recv_lvl(nlev, std::vector<long long>(nranks, 0));
    std::vector<HaloNeed> hn;
    std::vector<CrseNeed> cn;
    for (int l = 0; l < nlev; ++l) {
        const Level& V = lev[l];
        for (int gb = 0; gb < (int)V.boxes.size(); ++gb) {
            int downer = V.owner[gb];
            hn.clear();
            halo_needs_cross(*this, l, gb, hn, NEED_UNLINKED);     // linked faces are read in place, never exchanged
            for (auto& n : hn) {
                int sowner = V.owner[n.sbox];
                if (sowner == downer) continue;
                long long c = n.dst.npts();
                if (downer == rank) recv_lvl[l][sowner] += c;
                if (sowner == rank) {
                    Ent e; e.lev = l; e.peer = downer;
                    std::memset(&e.t, 0, sizeof(e.t));
                    e.t.sbox = V.g2l[n.sbox]; e.t.slev = l;
                    for (int d = 0; d < 3; ++d) { e.t.slo[d] = n.dst.lo[d] + n.shift[d]; e.t.n[d] = n.dst.len(d); }
                    sends.push_back(e);
                    send_lvl[l][downer] += c;
                }
            }
            if (l > 0) {
                const Level& C = lev[l - 1];
                for (int face = 0; face < 6; ++face) {
                    if (face_is_physical(*this, l, gb, face) || !face_has_uncovered(*this, l, gb, face)) continue;
                    cn.clear();
                    crse_needs(*this, l, gb, face, cn);
                    for (auto& n : cn) {
                        int sowner = C.owner[n.cbox];
                        // with peer links the coarse cells of another rank are read in place through the peer mapping
                        // (coarse gather index entries <= -3), like linked neighbour faces: nothing to exchange
                        if (sowner == downer || peer_links) continue;
                        long long c = n.reg.npts();
                        if (downer == rank) recv_lvl[l][sowner] += c;
                        if (sowner == rank) {
                            Ent e; e.lev = l; e.peer = downer;
                            std::memset(&e.t, 0, sizeof(e.t));
                            e.t.sbox = C.g2l[n.cbox]; e.t.slev = l - 1;
                            for (int d = 0; d < 3; ++d) { e.t.slo[d] = n.reg.lo[d] + n.shift[d]; e.t.n[d] = n.reg.len(d); }
                            sends.push_back(e);
                            send_lvl[l][downer] += c;
                        }
                    }
                }
            }
        }
    }
    // slab layout: per peer contiguous; inside a peer's block, fill levels ascending
    xplan.level_send_cell0.assign(nlev + 1, std::vector<long long>(nranks, 0));
    xplan.level_recv_cell0.assign(nlev + 1, std::vector<long long>(nranks, 0));
    long long so = 0, ro = 0;
    for (int p = 0; p < nranks; ++p) {
        xplan.send_prefix[p] = so; xplan.recv_prefix[p] = ro;
        for (int l = 0; l < nlev; ++l) {
            xplan.level_send_cell0[l][p] = so; so += send_lvl[l][p];
            xplan.level_recv_cell0[l][p] = ro; ro += recv_lvl[l][p];
        }
        xplan.level_send_cell0[nlev][p] = so;
        xplan.level_recv_cell0[nlev][p] = ro;
    }
    xplan.send_prefix[nranks] = so; xplan.recv_prefix[nranks] = ro;
    std::vector<std::vector<long long>> cur = xplan.level_send_cell0;
    xplan.pack.clear();
    xplan.pack_level_begin.assign(nlev + 1, 0);
    long long dense = 0;
    int curlev = 0;
    for (auto& e : sends) {
        while (curlev < e.lev) xplan.pack_level_begin[++curlev] = (long long)xplan.pack.size();
        e.t.dense = dense;
        e.t.start = cur[e.lev][e.peer];
        long long c = (long long)e.t.n[0] * e.t.n[1] * e.t.n[2];
        cur[e.lev][e.peer] += c;
        dense += c;
        xplan.pack.push_back(e.t);
    }
    while (curlev < nlev) xplan.pack_level_begin[++curlev] = (long long)xplan.pack.size();
    xplan.recv_ids.assign((size_t)xplan.recv_prefix[nranks], -1);
    xplan.send_ids.assign((size_t)xplan.send_prefix[nranks], -1);
    for (const PaPackTag& t : xplan.pack) {
        int gb = lev[t.slev].local[t.sbox];
        const Box& B = lev[t.slev].boxes[gb];
        long long q = 0;
        for (int k = 0; k < t.n[2]; ++k)
            for (int j = 0; j < t.n[1]; ++j)
                for (int i = 0; i < t.n[0]; ++i, ++q)
                    xplan.send_ids[(size_t)(t.start + q)] = cell_id(t.slev, gb, B, t.slo[0] + i, t.slo[1] + j, t.slo[2] + k);
    }
}

void Hier::build_halo(int l, int ng, bool cross, HaloTable& out, bool allow_remote) {
    const Level& V = lev[l];
    out.tags.clear();
    std::vector<PaHaloTag> remote;
    // receive cursors: position inside each peer's recv block.  Canonical order is level-major, so the cursor of
    // level l starts after everything levels < l receive from that peer (halo + coarse needs).  Recompute by replay.
    // receive cursors: position inside each peer's recv block for this fill level (canonical order: per dst box,
    // halo needs first, then its coarse needs)
    std::vector<long long> rcur;
    if (cross && allow_remote && nranks > 1) rcur = xplan.level_recv_cell0[l];
    std::vector<PaHaloTag> linked;
    if (cross) {
        std::vector<HaloNeed> hn; std::vector<CrseNeed> cn;
        for (int gb : V.local) {
            hn.clear();
            halo_needs_cross(*this, l, gb, hn, NEED_UNLINKED);
            for (auto& n : hn) {
                PaHaloTag t;
                std::memset(&t, 0, sizeof(t));
                t.dbox = V.g2l[gb];
                for (int d = 0; d < 3; ++d) { t.dlo[d] = n.dst.lo[d]; t.n[d] = n.dst.len(d); t.shift[d] = n.shift[d]; }
                int so = V.owner[n.sbox];
                t.srank = so;
                if (so == rank) { t.sbox = V.g2l[n.sbox]; t.rsrc = -1; out.tags.push_back(t); }
                else {
                    t.sbox = -1; t.rsrc = rcur[so]; rcur[so] += n.dst.npts(); remote.push_back(t);
                    const Box& SB = V.boxes[n.sbox];
                    long long q = 0;
                    for (int k = n.dst.lo[2]; k <= n.dst.hi[2]; ++k)
                        for (int j = n.dst.lo[1]; j <= n.dst.hi[1]; ++j)
                            for (int i = n.dst.lo[0]; i <= n.dst.hi[0]; ++i, ++q)
                                xplan.recv_ids[(size_t)(t.rsrc + q)] = cell_id(l, n.sbox, SB, i + n.shift[0], j + n.shift[1], k + n.shift[2]);
                }
            }
            // keep the per-peer cursor in canonical order: this box's coarse needs come next in the stream
            if (l > 0 && !rcur.empty())
                for (int face = 0; face < 6; ++face) {
                    if (face_is_physical(*this, l, gb, face) || !face_has_uncovered(*this, l, gb, face)) continue;
                    cn.clear(); crse_needs(*this, l, gb, face, cn);
                    for (auto& n : cn) if (!peer_links && lev[l - 1].owner[n.cbox] != rank) rcur[lev[l - 1].owner[n.cbox]] += n.reg.npts();
                }
            // linked faces: materialised only on request, straight from the neighbour (local or peer-mapped)
            hn.clear();
            halo_needs_cross(*this, l, gb, hn, NEED_LINKED);
            for (auto& n : hn) {
                PaHaloTag t;
                std::memset(&t, 0, sizeof(t));
                t.dbox = V.g2l[gb];
                for (int d = 0; d < 3; ++d) { t.dlo[d] = n.dst.lo[d]; t.n[d] = n.dst.len(d); t.shift[d] = n.shift[d]; }
                t.srank = V.owner[n.sbox];
                t.sbox = V.g2e[n.sbox];
                t.rsrc = -1;
                linked.push_back(t);
            }
        }
    } else {
        // full FillBoundary: grow(vbx, ng) + p against every box, minus vbx (AMReX_FabArrayBase.cpp:739-794)
        std::vector<std::array<int, 3>> sh;
        periodic_shifts(V.dom, ng, sh);
        std::vector<std::pair<int, Box>> is;
        std::vector<Box> parts;
        for (int gb : V.local) {
            Box grown = V.boxes[gb].grown(ng);
            for (auto& s : sh) {
                is.clear();
                V.hash.query(grown.shifted(s.data()), [&](int k, const Box& ib) { is.emplace_back(k, ib); });
                sort_isects(is);
                for (auto& e : is) {
                    if (V.owner[e.first] != rank) continue;        // several ranks: fill_patch's exchange moves these
                    int neg[3] = {-s[0], -s[1], -s[2]};
                    Box dst = e.second.shifted(neg);
                    parts.clear();
                    box_diff(dst, V.boxes[gb], parts);
                    for (Box& p : parts) {
                        PaHaloTag t;
                        std::memset(&t, 0, sizeof(t));
                        t.dbox = V.g2l[gb];
                        t.sbox = V.g2l[e.first];
                        t.srank = rank;
                        t.rsrc = -1;
                        for (int d = 0; d < 3; ++d) { t.dlo[d] = p.lo[d]; t.n[d] = p.len(d); t.shift[d] = s[d]; }
                        out.tags.push_back(t);
                    }
                }
            }
        }
    }
    out.nlocal_tags = (int)out.tags.size();
    out.tags.insert(out.tags.end(), remote.begin(), remote.end());
    out.ntags_unlinked = (int)out.tags.size();
    out.tags.insert(out.tags.end(), linked.begin(), linked.end());
    long long c = 0;
    out.ncells_unlinked = 0;
    for (size_t i = 0; i < out.tags.size(); ++i) {
        if ((int)i == out.ntags_unlinked) out.ncells_unlinked = c;
        PaHaloTag& t = out.tags[i];
        t.start = c; c += (long long)t.n[0] * t.n[1] * t.n[2];
    }
    if (out.ntags_unlinked == (int)out.tags.size()) out.ncells_unlinked = c;
    out.ncells = c;
}

const HaloTable& Hier::halo_full(int l, int ng) {
    auto key = std::make_pair(l, ng);
    auto it = halo_full_.find(key);
    if (it != halo_full_.end()) return it->second;
    HaloTable T;
    build_halo(l, ng, false, T, false);
    return halo_full_.emplace(key, std::move(T)).first->second;
}

// ---- filterPlt path: grids and FillPatch tables -------------------------------------------------------------------
// BoxList::maxSize (AMReX_BoxList.cpp:765-815): per direction the length and the chunk are divided by their common powers
// of two, the coarsened length is cut into ceil(nlen / bs) blocks whose sizes differ by at most one (the larger ones
// first), and the blocks are scaled back; the chunks of a box replace it in place, x fastest.
void box_max_size(int nboxes, const int* boxes, int max_grid_size, std::vector<Box>& out) {
    out.clear();
    for (int b = 0; b < nboxes; ++b) {
        Box bx;
        for (int d = 0; d < 3; ++d) { bx.lo[d] = boxes[6 * b + d]; bx.hi[d] = boxes[6 * b + 3 + d]; }
        int ratio[3] = {1, 1, 1}, numblk[3] = {1, 1, 1}, extra[3] = {0, 0, 0}, sz[3];
        for (int d = 0; d < 3; ++d) {
            sz[d] = bx.len(d);
            if (bx.len(d) > max_grid_size) {
                int bs = max_grid_size, nlen = bx.len(d);
                while (bs % 2 == 0 && nlen % 2 == 0) { ratio[d] *= 2; bs /= 2; nlen /= 2; }
                numblk[d] = (nlen + bs - 1) / bs;
                sz[d] = nlen / numblk[d];
                extra[d] = nlen - sz[d] * numblk[d];
            }
        }
        auto cut = [&](int d, int a, int& l0, int& h0) {
            if (a < extra[d]) { l0 = a * (sz[d] + 1) * ratio[d]; h0 = l0 + (sz[d] + 1) * ratio[d] - 1; }
            else { l0 = (a * sz[d] + extra[d]) * ratio[d]; h0 = l0 + sz[d] * ratio[d] - 1; }
            l0 += bx.lo[d]; h0 += bx.lo[d];
        };
        if (numblk[0] == 1 && numblk[1] == 1 && numblk[2] == 1) { out.push_back(bx); continue; }
        for (int k = 0; k < numblk[2]; ++k)
            for (int j = 0; j < numblk[1]; ++j)
                for (int i = 0; i < numblk[0]; ++i) {
                    Box c;
                    cut(0, i, c.lo[0], c.hi[0]); cut(1, j, c.lo[1], c.hi[1]); cut(2, k, c.lo[2], c.hi[2]);
                    out.push_back(c);
                }
    }
}

// FillPatchTwoLevels as filterPlt calls it (filterPlt.cpp:170-203; FabArrayBase::FPinfo): for every local box the part of
// its grown region that lies inside the domain and that no box of the level covers is cut into boxes ("pieces",
// BoxArray::complementIn); each piece is interpolated from a coarse patch that is gathered from the coarse level's valid
// cells.  Ghost cells outside the (non-periodic) domain are first-order extrapolated afterwards: `clamps`.
// On several ranks the walk goes over every box of the level (global id order): a source owned by the destination box's
// owner is a local table entry there, any other source joins the slab stream (source owner -> destination owner), which the
// source's owner packs (`pack`) and the destination's owner unpacks (`unpack`) -- what ParallelCopy / FillBoundary
// communicate inside FillPatchTwoLevels.
const FillPatchTable& Hier::fill_patch(int l, int ng, int cgrow) {
    std::array<int, 3> key{l, ng, cgrow};
    auto it = fill_patch_.find(key);
    if (it != fill_patch_.end()) return it->second;
    FillPatchTable T;
    const Level& V = lev[l];
    struct XSend { int peer; PaPackTag t; };
    struct XRecv { int peer; int slev, sgb; PaFpUnpack u; };
    std::vector<XSend> xs;
    std::vector<XRecv> xr;
    // a source region (index space of level slev, cells [r.lo, r.hi]) of global box sgb for destination `dst` (>= 0: local
    // fine box, < 0: piece) of a box owned by `downer`
    auto cross = [&](int downer, int slev, int sgb, const Box& r, int dst) {
        const int sowner = lev[slev].owner[sgb];
        if (downer == rank) {
            XRecv e; e.peer = sowner; e.slev = slev; e.sgb = sgb;
            std::memset(&e.u, 0, sizeof(e.u));
            e.u.box = dst;
            for (int d = 0; d < 3; ++d) { e.u.lo[d] = r.lo[d]; e.u.n[d] = r.len(d); }
            xr.push_back(e);
        } else if (sowner == rank) {
            XSend e; e.peer = downer;
            std::memset(&e.t, 0, sizeof(e.t));
            e.t.sbox = lev[slev].g2l[sgb]; e.t.slev = slev;
            for (int d = 0; d < 3; ++d) { e.t.slo[d] = r.lo[d]; e.t.n[d] = r.len(d); }
            xs.push_back(e);
        }
    };
    for (size_t lb = 0; lb < V.local.size(); ++lb) {
        const Box g = V.boxes[V.local[lb]].grown(ng);
        bool out = false;
        for (int d = 0; d < 3; ++d) out |= g.lo[d] < V.dom.lo[d] || g.hi[d] > V.dom.hi[d];
        if (out) {
            PaFpClamp c;
            c.box = (int)lb; c.pad = 0; c.start = T.nclamp;
            T.nclamp += g.npts();
            T.clamps.push_back(c);
        }
    }
    // one rank: the local boxes are all boxes, in the same order
    const std::vector<int> every = [&] { std::vector<int> v(V.boxes.size()); for (size_t b = 0; b < v.size(); ++b) v[b] = (int)b; return v; }();
    const std::vector<int>& walk = nranks > 1 ? every : V.local;
    std::vector<std::pair<int, Box>> is;
    std::vector<Box> parts;
    const Level* Cv = l > 0 ? &lev[l - 1] : nullptr;
    std::vector<Box> cur, nxt;
    for (int gb : walk) {
        const int downer = V.owner[gb];
        const bool mine = downer == rank;
        // 1. same-level sources of another rank, in halo_full's order (grown(ng) against every box, minus the own box)
        if (nranks > 1) {
            is.clear();
            V.hash.query(V.boxes[gb].grown(ng), [&](int k, const Box& ib) { is.emplace_back(k, ib); });
            sort_isects(is);
            for (auto& e : is) {
                if (V.owner[e.first] == downer) continue;
                parts.clear();
                box_diff(e.second, V.boxes[gb], parts);
                for (const Box& p : parts) cross(downer, l, e.first, p, mine ? V.g2l[gb] : 0);
            }
        }
        if (!Cv) continue;
        // 2. coarse patches of the pieces
        const int r = V.ratio;
        const Box region = V.boxes[gb].grown(ng).isect(V.dom);
        cur.assign(1, region);
        V.hash.query(region, [&](int idx, const Box&) {
            nxt.clear();
            for (const Box& b : cur) box_diff(b, V.boxes[idx], nxt);
            cur.swap(nxt);
        });
        for (const Box& pc : cur) {
            PaFpPiece P;
            P.box = mine ? V.g2l[gb] : -1;
            Box cp;
            for (int d = 0; d < 3; ++d) {
                P.lo[d] = pc.lo[d]; P.n[d] = pc.len(d);
                cp.lo[d] = coarsen(pc.lo[d], r) - cgrow; cp.hi[d] = coarsen(pc.hi[d], r) + cgrow;
                P.clo[d] = cp.lo[d]; P.cn[d] = cp.len(d);
            }
            P.cstart = T.ncrse; P.fstart = T.nfine;
            const Box cpd = cp.isect(Cv->dom);
            long long got = 0;
            const int piece = (int)T.pieces.size();
            Cv->hash.query(cpd, [&](int idx, const Box& ib) {
                got += ib.npts();
                if (Cv->owner[idx] != downer) { cross(downer, l - 1, idx, ib, -1 - piece); return; }
                if (!mine) return;
                PaFpCopy c;
                c.piece = piece; c.sbox = Cv->g2l[idx];
                for (int d = 0; d < 3; ++d) { c.lo[d] = ib.lo[d]; c.n[d] = ib.len(d); }
                c.start = T.ncopy;
                T.ncopy += ib.npts();
                T.copies.push_back(c);
            });
            if (got != cpd.npts() && T.err.empty())
                T.err = "level " + std::to_string(l) + ": ghost cells of box " + std::to_string(gb) +
                        " need coarse cells that level " + std::to_string(l - 1) + " does not cover (grids not properly nested for this ghost width)";
            if (!mine) continue;
            T.ncrse += cp.npts(); T.nfine += pc.npts();
            T.pieces.push_back(P);
        }
    }
    if (nranks > 1) {
        // slab layout: per peer contiguous, walk order inside a peer's block
        T.send_prefix.assign(nranks + 1, 0);
        T.recv_prefix.assign(nranks + 1, 0);
        for (const XSend& e : xs) T.send_prefix[e.peer + 1] += (long long)e.t.n[0] * e.t.n[1] * e.t.n[2];
        for (const XRecv& e : xr) T.recv_prefix[e.peer + 1] += (long long)e.u.n[0] * e.u.n[1] * e.u.n[2];
        for (int p = 0; p < nranks; ++p) { T.send_prefix[p + 1] += T.send_prefix[p]; T.recv_prefix[p + 1] += T.recv_prefix[p]; }
        std::vector<long long> sc(T.send_prefix.begin(), T.send_prefix.end() - 1), rc(T.recv_prefix.begin(), T.recv_prefix.end() - 1);
        T.send_ids.assign((size_t)T.send_prefix[nranks], -1);
        T.recv_ids.assign((size_t)T.recv_prefix[nranks], -1);
        auto ids = [&](std::vector<long long>& out, long long at, int slev, int sgb, const int* lo, const int* n) {
            const Box& B = lev[slev].boxes[sgb];
            long long q = 0;
            for (int k = 0; k < n[2]; ++k)
                for (int j = 0; j < n[1]; ++j)
                    for (int i = 0; i < n[0]; ++i, ++q) out[(size_t)(at + q)] = cell_id(slev, sgb, B, lo[0] + i, lo[1] + j, lo[2] + k);
        };
        for (XSend& e : xs) {
            const long long c = (long long)e.t.n[0] * e.t.n[1] * e.t.n[2];
            e.t.dense = T.npack; e.t.start = sc[e.peer];
            ids(T.send_ids, e.t.start, e.t.slev, lev[e.t.slev].local[e.t.sbox], e.t.slo, e.t.n);
            sc[e.peer] += c; T.npack += c;
            T.pack.push_back(e.t);
        }
        for (XRecv& e : xr) {
            const long long c = (long long)e.u.n[0] * e.u.n[1] * e.u.n[2];
            e.u.start = T.nunpack; e.u.rsrc = rc[e.peer];
            ids(T.recv_ids, e.u.rsrc, e.slev, e.sgb, e.u.lo, e.u.n);
            rc[e.peer] += c; T.nunpack += c;
            T.unpack.push_back(e.u);
        }
    }
    return fill_patch_.emplace(key, std::move(T)).first->second;
}

// poly_interp_coeff (AMReX_LOUtil_K.H:24-37), same loop so the last bits match
static void poly_interp_coeff(double xInt, const double* x, int N, double* c) {
    for (int j = 0; j < N; ++j) {
        double num = 1.0, den = 1.0;
        for (int i = 0; i < N; ++i)
            if (i != j) { num *= xInt - x[i]; den *= x[j] - x[i]; }
        c[j] = num / den;
    }
}

std::string Hier::build_faces() {
    // level 0 must cover the domain.  Decided over every box of the level, not only this rank's, so that on several ranks
    // every rank rejects the same hierarchy before any communication (the same first box, hence the same message, as the
    // per-record check below finds on one rank).
    for (int gb = 0; gb < (int)lev[0].boxes.size(); ++gb)
        for (int face = 0; face < 6; ++face)
            if (!face_is_physical(*this, 0, gb, face) && face_has_uncovered(*this, 0, gb, face))
                return "level 0 does not cover the domain (box " + std::to_string(gb) + " has an interior face with no neighbour)";
    faces = FaceTable();
    faces.level_rec_begin.assign(nlev + 1, 0);
    std::vector<uint8_t> m;
    std::vector<CrseNeed> cn;
    // receive cursors for the coarse needs (canonical order, see build_exchange)
    std::vector<long long> rcur;
    std::vector<HaloNeed> hn;
    for (int l = 0; l < nlev; ++l) {
        const Level& V = lev[l];
        if (nranks > 1) rcur = xplan.level_recv_cell0[l];
        faces.level_rec_begin[l] = (long long)faces.recs.size();
        const int r = V.ratio;
        const int E = (l > 0) ? r : 0;                       // tangential reach of the o3 stencil's mask tests
        for (int gb : V.local) {
            const Box& B = V.boxes[gb];
            if (nranks > 1) {                                // this box's halo needs precede its coarse needs in the stream
                hn.clear(); halo_needs_cross(*this, l, gb, hn, NEED_UNLINKED);
                for (auto& n : hn) if (V.owner[n.sbox] != rank) rcur[V.owner[n.sbox]] += n.dst.npts();
            }
            for (int face = 0; face < 6; ++face) {
                const int d = face % 3;
                const int t1 = (d == 0) ? 1 : 0, t2 = (d == 2) ? 1 : 2;
                const bool physical = face_is_physical(*this, l, gb, face);
                if (!physical && !face_has_uncovered(*this, l, gb, face)) continue;
                // mask plane grown tangentially by E.  Domain grown by 5 in periodic directions for the BndryData
                // mask (NTangHalfWidth) and by 1 for m_maskvals: identical on every cell consulted here because
                // tangential offsets never exceed the ratio (<=4) and the normal offset is 1.
                Box plane = face_plane(B, face, 1, E);
                plane_mask(*this, l, plane, 5, m);
                int pn[3] = {plane.len(0), plane.len(1), plane.len(2)};
                auto M = [&](int a1, int a2) -> int {        // a1,a2 offsets from B.lo along t1,t2 (may be negative)
                    int c[3];
                    c[d] = 0; c[t1] = a1 + E; c[t2] = a2 + E;
                    return m[((size_t)c[2] * pn[1] + c[1]) * pn[0] + c[0]];
                };
                PaFaceRec R;
                std::memset(&R, 0, sizeof(R));
                R.box = V.g2l[gb]; R.face = face; R.ratio = r;
                R.n1 = B.len(t1); R.n2 = B.len(t2);
                R.start = (long long)faces.flags.size();
                R.cidx = -1;
                bool any = false;
                for (int a2 = 0; a2 < R.n2; ++a2)
                    for (int a1 = 0; a1 < R.n1; ++a1) {
                        unsigned f = (unsigned)M(a1, a2);
                        if (f) any = true;
                        if (l > 0) {
                            static const int o1[8] = {-1, 1, 0, 0, -1, 1, -1, 1};
                            static const int o2[8] = {0, 0, -1, 1, -1, -1, 1, 1};
                            for (int b = 0; b < 8; ++b)
                                if (M(a1 + o1[b] * r, a2 + o2[b] * r) == 1) f |= 1u << (2 + b);
                        }
                        faces.flags.push_back((uint16_t)f);
                    }
                if (!any) { faces.flags.resize((size_t)R.start); continue; }
                if (physical) {
                    R.kind = (bc_kind[d] == 1) ? PA_FACE_REFLECT_ODD : PA_FACE_NEUMANN;
                    R.nx = 1;
                } else {
                    if (l == 0) return "level 0 does not cover the domain (box " + std::to_string(gb) + " has an interior face with no neighbour)";
                    R.kind = PA_FACE_CF;
                    int blen = B.len(d);
                    R.nx = std::min(blen + 1, 4);
                    double bcl = 0.5 * (double)r * V.dx[d];              // AMReX_MLMGBndry.H:146-148
                    double x[4] = {-bcl * V.dxinv[d], 0.5, 1.5, 2.5};    // AMReX_MLLinOp_K.H:51
                    poly_interp_coeff(-0.5, x, R.nx, R.coef);
                    Box rb = crse_register_box(B, r, face);
                    R.rlo1 = rb.lo[t1]; R.rlo2 = rb.lo[t2];
                    R.rn1 = rb.len(t1); R.rn2 = rb.len(t2);
                    R.cidx = (long long)faces.cidx.size();
                    PaCrseIdx none; none.box = -1; none.rel = 0;
                    faces.cidx.resize(faces.cidx.size() + (size_t)R.rn1 * R.rn2, none);
                    cn.clear();
                    crse_needs(*this, l, gb, face, cn);
                    const Level& C = lev[l - 1];
                    for (auto& n : cn) {
                        const Box& cb = C.boxes[n.cbox];
                        bool local = (C.owner[n.cbox] == rank);
                        const bool in_place = !local && peer_links;     // a peer's coarse box, read through the peer mapping
                        long long rbase = 0;
                        if (!local && !in_place) { rbase = rcur[C.owner[n.cbox]]; rcur[C.owner[n.cbox]] += n.reg.npts(); }
                        long long q = 0;
                        for (int k = n.reg.lo[2]; k <= n.reg.hi[2]; ++k)
                            for (int j = n.reg.lo[1]; j <= n.reg.hi[1]; ++j)
                                for (int i = n.reg.lo[0]; i <= n.reg.hi[0]; ++i, ++q) {
                                    int c[3] = {i, j, k};
                                    size_t e = (size_t)R.cidx + (size_t)(c[t2] - R.rlo2) * R.rn1 + (size_t)(c[t1] - R.rlo1);
                                    PaCrseIdx& X = faces.cidx[e];
                                    if (local || in_place) {
                                        X.box = local ? C.g2l[n.cbox] : -3 - n.cbox;        // <= -3: GLOBAL id of a peer-owned box
                                        X.rel = (unsigned)(i + n.shift[0] - cb.lo[0]) | ((unsigned)(j + n.shift[1] - cb.lo[1]) << 10) |
                                                ((unsigned)(k + n.shift[2] - cb.lo[2]) << 20);
                                    } else {
                                        X.box = -2;
                                        X.rel = (unsigned)(rbase + q);
                                        xplan.recv_ids[(size_t)(rbase + q)] = cell_id(l - 1, n.cbox, cb, i + n.shift[0], j + n.shift[1], k + n.shift[2]);
                                    }
                                }
                    }
                }
                faces.recs.push_back(R);
                faces.rec_level.push_back(l);
            }
        }
    }
    faces.level_rec_begin[nlev] = (long long)faces.recs.size();
    faces.ncells = (long long)faces.flags.size();
    faces.level_blk_begin.assign(nlev + 1, 0);
    for (int l = 0; l < nlev; ++l) {
        faces.level_blk_begin[l] = (long long)faces.blocks.size();
        for (long long r = faces.level_rec_begin[l]; r < faces.level_rec_begin[l + 1]; ++r) {
            const int n = faces.recs[r].n1 * faces.recs[r].n2;
            for (int c = 0; c < n; c += PA_FACE_CHUNK) faces.blocks.push_back(PaFaceBlock{(int)r, c});
        }
    }
    faces.level_blk_begin[nlev] = (long long)faces.blocks.size();
    return "";
}

std::vector<long long> Hier::crse_offsets(int ng) {
    std::vector<long long> out(faces.cidx.size(), -1);
    for (size_t r = 0; r < faces.recs.size(); ++r) {
        const PaFaceRec& R = faces.recs[r];
        if (R.cidx < 0) continue;
        const Layout& Y = layout(faces.rec_level[r] - 1, ng);
        const long long n = (long long)R.rn1 * R.rn2;
        for (long long e = R.cidx; e < R.cidx + n; ++e) {
            const PaCrseIdx& X = faces.cidx[(size_t)e];
            if (X.box >= 0) {
                const PaLayDev& y = Y.lay[X.box];
                const int i = (int)(X.rel & 1023u), j = (int)((X.rel >> 10) & 1023u), k = (int)(X.rel >> 20);
                out[(size_t)e] = y.off + (long long)(k + y.ng) * y.PS + (long long)(j + y.ng) * y.P + (i + y.ng + y.xoff);
            } else if (X.box == -1) {
                out[(size_t)e] = -1;
            } else if (X.box == -2) {
                out[(size_t)e] = -2 - (long long)X.rel;
            } else {
                // peer-owned coarse box: (owner rank, element offset inside that rank's slab), PA_CRSE_PEER_* in pa_types.h
                const int gid = -3 - X.box;
                const PaLayDev& y = Y.all[(size_t)gid];
                const int i = (int)(X.rel & 1023u), j = (int)((X.rel >> 10) & 1023u), k = (int)(X.rel >> 20);
                const long long off = y.off + (long long)(k + y.ng) * y.PS + (long long)(j + y.ng) * y.P + (i + y.ng + y.xoff);
                out[(size_t)e] = -(PA_CRSE_PEER_BASE + ((long long)lev[faces.rec_level[r] - 1].owner[gid] << PA_CRSE_PEER_SHIFT) + off);
            }
        }
    }
    return out;
}

// Order the boxes along a curve through their low corners and cut the curve into nranks chunks of ~equal cell volume
// (the idea of DistributionMapping::SFCProcessorMap, AMReX_DistributionMapping.cpp:1262-1320; any box -> rank map is valid).
// Default curve: lexicographic in (z, y, x) -- x fastest.  A chunk is then a run of whole x-rows of boxes (z-slabs, cut in y
// where a slab holds more than one rank), so a rank boundary is a y or z face wherever the level has at least one x-row of
// boxes per rank: cross-rank ghost data then moves as whole contiguous rows / planes (one TMA bulk copy over NVLink each),
// never as the per-row 8-byte column loads an x face costs (round 1: the Morton curve cut x at 8 ranks and the
// efficiency fell from 0.95 to 0.81 there).  PA_DISTRIBUTE=morton selects the Morton curve (x in the lowest bit).
void sfc_distribute(int nboxes, const int* boxes, int nranks, int* owner_out) {
    std::vector<std::pair<uint64_t, int>> keys(nboxes);
    int mn[3] = {1 << 30, 1 << 30, 1 << 30};
    for (int b = 0; b < nboxes; ++b)
        for (int d = 0; d < 3; ++d) mn[d] = std::min(mn[d], boxes[6 * b + d]);
    const char* ecurve = getenv("PA_DISTRIBUTE");
    const bool morton = ecurve && !strcmp(ecurve, "morton");
    auto spread = [morton](uint64_t v) {
        uint64_t x = v & 0x1fffff;
        if (!morton) return x;
        x = (x | x << 32) & 0x1f00000000ffffULL;
        x = (x | x << 16) & 0x1f0000ff0000ffULL;
        x = (x | x << 8) & 0x100f00f00f00f00fULL;
        x = (x | x << 4) & 0x10c30c30c30c30c3ULL;
        x = (x | x << 2) & 0x1249249249249249ULL;
        return x;
    };
    double total = 0;
    for (int b = 0; b < nboxes; ++b) {
        uint64_t k = 0;
        for (int d = 0; d < 3; ++d) k |= spread((uint64_t)(boxes[6 * b + d] - mn[d])) << (morton ? d : 21 * d);
        keys[b] = {k, b};
        double v = 1;
        for (int d = 0; d < 3; ++d) v *= boxes[6 * b + 3 + d] - boxes[6 * b + d] + 1;
        total += v;
    }
    std::sort(keys.begin(), keys.end());
    double acc = 0;
    for (auto& kb : keys) {
        int b = kb.second;
        double v = 1;
        for (int d = 0; d < 3; ++d) v *= boxes[6 * b + 3 + d] - boxes[6 * b + d] + 1;
        int r = (int)std::floor((acc + 0.5 * v) / total * nranks);
        owner_out[b] = std::min(std::max(r, 0), nranks - 1);
        acc += v;
    }
}

// Tables of pa_smooth's composite operator (see DESIGN.md section 10):
//  * the box-face records with the coarse-fine polynomial of order `maxorder` (the halo tables, masks and coarse gather
//    indices of faces are shared with every other ghost fill; only NX and the coefficients differ);
//  * the covered coarse cells of every level, per (coarse box, fine box) intersection (average_down);
//  * the coarse side of every coarse-fine face (reflux), one record per coarse face, found from the fine level's
//    coarse-fine ghost cells (mask not_covered on a coarse-fine face record), periodic images included.
const SmoothTables& Hier::smooth_tables(int maxorder) {
    auto it = smooth_.find(maxorder);
    if (it != smooth_.end()) return it->second;
    SmoothTables T;
    auto done = [&]() -> const SmoothTables& { return smooth_.emplace(maxorder, std::move(T)).first->second; };
    if (nranks > 1) { T.err = "pa_smooth supports one rank only"; return done(); }
    if (filter_only) { T.err = "pa_smooth needs a hierarchy created without PA_HIER_FILTER_ONLY"; return done(); }
    for (int l = 1; l < nlev; ++l)
        if (lev[l].ratio != 2) {
            T.err = "pa_smooth supports refinement ratio 2 only (level " + std::to_string(l) + " has ratio " + std::to_string(lev[l].ratio) +
                    "; curvature.cpp hard-codes 2)";
            return done();
        }
    T.recs = faces.recs;
    for (size_t q = 0; q < T.recs.size(); ++q) {
        PaFaceRec& R = T.recs[q];
        if (R.kind != PA_FACE_CF) continue;
        const Level& V = lev[faces.rec_level[q]];
        const int d = R.face % 3;
        const Box& B = V.boxes[V.local[R.box]];
        R.nx = std::min(B.len(d) + 1, maxorder);
        double bcl = 0.5 * (double)R.ratio * V.dx[d];
        double x[4] = {-bcl * V.dxinv[d], 0.5, 1.5, 2.5};
        for (int m = 0; m < 4; ++m) R.coef[m] = 0.0;
        poly_interp_coeff(-0.5, x, R.nx, R.coef);
    }
    T.avg_begin.assign(nlev + 1, 0);
    T.avg_cells.assign(nlev, 0);
    for (int lc = 0; lc < nlev; ++lc) {
        T.avg_begin[lc] = (long long)T.avg.size();
        if (lc + 1 >= nlev) continue;
        const Level& C = lev[lc];
        const Level& F = lev[lc + 1];
        long long start = 0;
        for (int fg : F.local) {
            Box cb = F.boxes[fg];
            for (int d = 0; d < 3; ++d) { cb.lo[d] = coarsen(cb.lo[d], 2); cb.hi[d] = coarsen(cb.hi[d], 2); }
            std::vector<std::pair<int, Box>> is;
            C.hash.query(cb, [&](int k, const Box& ib) { is.emplace_back(k, ib); });
            std::sort(is.begin(), is.end(), [](const std::pair<int, Box>& a, const std::pair<int, Box>& b) { return a.first < b.first; });
            for (auto& e : is) {
                PaAvgDown A;
                A.cbox = C.g2l[e.first]; A.fbox = F.g2l[fg];
                for (int d = 0; d < 3; ++d) { A.lo[d] = e.second.lo[d]; A.n[d] = e.second.len(d); }
                A.start = start;
                start += e.second.npts();
                T.avg.push_back(A);
            }
        }
        T.avg_cells[lc] = start;
    }
    T.avg_begin[nlev] = (long long)T.avg.size();
    std::map<std::array<int, 7>, PaReflux> rf;            // (coarse level, dir, side, coarse box, c[2], c[1], c[0])
    for (int lf = 1; lf < nlev; ++lf) {
        const Level& F = lev[lf];
        const Level& C = lev[lf - 1];
        for (long long q = faces.level_rec_begin[lf]; q < faces.level_rec_begin[lf + 1]; ++q) {
            const PaFaceRec& R = faces.recs[q];
            if (R.kind != PA_FACE_CF) continue;
            const int gb = F.local[R.box];
            const Box& B = F.boxes[gb];
            const int d = R.face % 3;
            const int t1 = (d == 0) ? 1 : 0, t2 = (d == 2) ? 1 : 2;
            const bool lo_face = R.face < 3;
            for (int a2 = 0; a2 < R.n2; ++a2)
                for (int a1 = 0; a1 < R.n1; ++a1) {
                    if (PA_FLAG_MASK(faces.flags[R.start + (long long)a2 * R.n1 + a1]) != 1) continue;
                    int g[3];
                    g[d] = lo_face ? B.lo[d] - 1 : B.hi[d] + 1;
                    g[t1] = B.lo[t1] + a1; g[t2] = B.lo[t2] + a2;
                    int w[3] = {g[0], g[1], g[2]};
                    const int nd = F.dom.len(d);
                    if (w[d] < F.dom.lo[d]) { if (!is_per[d]) continue; w[d] += nd; }
                    if (w[d] > F.dom.hi[d]) { if (!is_per[d]) continue; w[d] -= nd; }
                    int cc[3];
                    for (int e = 0; e < 3; ++e) cc[e] = coarsen(w[e], 2);
                    int cg = -1;
                    Box one{{cc[0], cc[1], cc[2]}, {cc[0], cc[1], cc[2]}};
                    C.hash.query(one, [&](int k, const Box&) { cg = k; });
                    if (cg < 0) {
                        T.err = "pa_smooth: level " + std::to_string(lf) + " is not properly nested in level " + std::to_string(lf - 1) +
                                " (a coarse-fine face of box " + std::to_string(gb) + " has no coarse cell)";
                        return done();
                    }
                    const Box& CB = C.boxes[cg];
                    const int side = lo_face ? 1 : 0;
                    std::array<int, 7> key{lf - 1, d, side, C.g2l[cg], cc[2] - CB.lo[2], cc[1] - CB.lo[1], cc[0] - CB.lo[0]};
                    if (rf.count(key)) continue;
                    PaReflux X;
                    X.cbox = C.g2l[cg]; X.fbox = R.box; X.dir = d; X.side = side;
                    for (int e = 0; e < 3; ++e) X.c[e] = cc[e] - CB.lo[e];
                    X.f[d] = (lo_face ? B.lo[d] : B.hi[d]) - B.lo[d];
                    X.f[t1] = 2 * coarsen(g[t1], 2) - B.lo[t1];
                    X.f[t2] = 2 * coarsen(g[t2], 2) - B.lo[t2];
                    rf.emplace(key, X);
                }
        }
    }
    T.reflux_begin.assign((size_t)nlev * 6 + 1, 0);
    for (auto& kv : rf) {
        T.reflux.push_back(kv.second);
        ++T.reflux_begin[(size_t)kv.first[0] * 6 + 2 * kv.first[1] + kv.first[2] + 1];
    }
    for (size_t i = 1; i < T.reflux_begin.size(); ++i) T.reflux_begin[i] += T.reflux_begin[i - 1];
    // coarsenings of level 0 for the multigrid preconditioner (one rank: local index = global id)
    T.mg_boxes.push_back(lev[0].boxes);
    T.mg_dom.push_back(lev[0].dom);
    T.mg_avg_begin.push_back(0);
    auto coarsenable = [](const Box& B) {
        for (int d = 0; d < 3; ++d)
            if ((B.lo[d] & 1) || (B.len(d) & 1) || B.len(d) < 4) return false;
        return true;
    };
    auto half = [](const Box& B) {
        Box c;
        for (int d = 0; d < 3; ++d) { c.lo[d] = B.lo[d] / 2; c.hi[d] = (B.hi[d] + 1) / 2 - 1; }
        return c;
    };
    for (;;) {
        const std::vector<Box>& F = T.mg_boxes.back();
        if (!coarsenable(T.mg_dom.back()) || !std::all_of(F.begin(), F.end(), coarsenable)) break;
        std::vector<Box> C(F.size());
        long long start = 0;
        for (size_t b = 0; b < F.size(); ++b) {
            C[b] = half(F[b]);
            PaAvgDown A;
            A.cbox = A.fbox = (int)b;
            for (int d = 0; d < 3; ++d) { A.lo[d] = C[b].lo[d]; A.n[d] = C[b].len(d); }
            A.start = start;
            start += C[b].npts();
            T.mg_avg.push_back(A);
        }
        T.mg_avg_cells.push_back(start);
        T.mg_avg_begin.push_back((long long)T.mg_avg.size());
        T.mg_dom.push_back(half(T.mg_dom.back()));
        T.mg_boxes.push_back(std::move(C));
    }
    return done();
}

}  // namespace pa
