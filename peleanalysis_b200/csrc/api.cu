// api.cu -- implementation of the C ABI declared in include/pele_stencil_b200.h.
// Host logic only: owns device memory, uploads the descriptor tables built by hier.cpp, sequences kernel launches.
// There is no CPU compute fallback anywhere in this file: without a usable device every compute call fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/pele_stencil_b200.h"
#include "hier.hpp"
#include "kernels.cuh"

using namespace pa;

namespace pa {
namespace {
std::mutex g_alloc_mu;
std::map<void*, std::pair<int, size_t>> g_alloc;       // live allocation -> (device, bytes)
std::map<int, int64_t> g_alloc_bytes;                  // device -> live bytes
}  // namespace

cudaError_t dev_alloc(void** p, size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lk(g_alloc_mu);
    g_alloc[*p] = {dev, bytes};
    g_alloc_bytes[dev] += (int64_t)bytes;
    return cudaSuccess;
}
void dev_free(void* p) {
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(g_alloc_mu);
        auto it = g_alloc.find(p);
        if (it != g_alloc.end()) {
            g_alloc_bytes[it->second.first] -= (int64_t)it->second.second;
            g_alloc.erase(it);
        }
    }
    cudaFree(p);
}
}  // namespace pa

namespace {

thread_local std::string t_err;
thread_local cudaStream_t t_stream = nullptr;

int fail(int code, const std::string& msg) { t_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
    return fail(PA_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
std::atomic<long long> g_fused_launches{0};
#define CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return cuda_fail(e__, #call); } while (0)
#define CHK(call) do { int r__ = (call); if (r__ != PA_OK) return r__; } while (0)

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    ~DevBuf() { if (p) dev_free(p); }
    cudaError_t upload(const std::vector<T>& v, cudaStream_t st) {
        if (p) { dev_free(p); p = nullptr; }
        n = v.size();
        if (!n) return cudaSuccess;
        cudaError_t e = dev_alloc((void**)&p, n * sizeof(T));
        if (e != cudaSuccess) return e;
        return cudaMemcpyAsync(p, v.data(), n * sizeof(T), cudaMemcpyHostToDevice, st);
    }
    cudaError_t reserve(size_t m) {
        if (m <= n) return cudaSuccess;
        if (p) { dev_free(p); p = nullptr; n = 0; }
        cudaError_t e = dev_alloc((void**)&p, m * sizeof(T));
        if (e == cudaSuccess) n = m;
        return e;
    }
};

struct LevelDev {
    DevBuf<PaBoxDev> boxes;                            // extended index (local boxes, then peer-owned link targets)
    DevBuf<PaNbr> nbr;                                 // neighbour links of the local boxes
    DevBuf<PaHaloTag> halo_cross;
    DevBuf<long long> host_off;                        // nlocal+1 prefix of valid cells (host concat order)
    DevBuf<int> gid;                                   // global box id of every local box
    std::vector<long long> host_off_h;
    // device-array copies (pa_field_upload_device): row items of the local boxes and the lanes per row, built on first use
    std::vector<PaRowItem> io_items_h;
    DevBuf<PaRowItem> io_items;
    int io_lg_s = 0;
};

// Tiles are stored class-major, level-minor: a "class" groups the boxes one CTA shape of the TMA pipeline serves
// (x-pairs per tile plane <= 128, <= 256, more), so a stencil pass over levels [l0, l1] is one contiguous tile range --
// one launch -- per class that occurs, each in the shape that fits its tiles.  The simple kernel has one class.
constexpr int N_TILE_CLASSES = 3;
struct TileTable {
    std::vector<PaTile> h;
    DevBuf<PaTile> d;
    long long begin[N_TILE_CLASSES][PA_MAX_LEVELS + 1];        // first tile of (class, level); [c][nlev] = end of the class
    int plane_doubles[N_TILE_CLASSES][PA_MAX_LEVELS];          // largest staged plane (ng = 1 input layout, one component)
    int items[N_TILE_CLASSES][PA_MAX_LEVELS];                  // most x-pairs per tile plane
    int max_plane_doubles = 0;                                 // over all tiles
    bool ok = true;
};

// pa_smooth: the composite operator's tables on the device and the solver's work fields (allocated on the first call)
struct SmoothDev {
    DevBuf<PaFaceRec> recs;                            // face records with the smoothing operator's coarse-fine polynomial
    DevBuf<PaAvgDown> avg;
    DevBuf<PaReflux> reflux;
    DevBuf<double> partial, scal;                      // reduction partials and the reduced scalar
    pa_field* w[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // multigrid preconditioner (built on the first PA_SMOOTH_PRECOND_MG call): the V-cycle's right-hand side and residual on
    // the hierarchy, and the coarsenings of level 0 (MG levels 1, 2, ...) as single-level one-rank hierarchies with their
    // correction, right-hand side and residual fields
    pa_field* mg_rhs = nullptr;
    pa_field* mg_res = nullptr;
    std::vector<pa_hier*> mg_h;
    std::vector<std::array<pa_field*, 3>> mg_f;
    DevBuf<PaAvgDown> mg_avg;
    bool mg_ready = false;
};

}  // namespace

struct pa_hier {
    Hier H;
    bool dev_ready = false;
    std::vector<std::unique_ptr<LevelDev>> lev;
    std::map<std::pair<int, int>, std::unique_ptr<DevBuf<PaLayDev>>> lay;         // (level, ng)
    std::map<std::pair<int, int>, std::unique_ptr<DevBuf<PaHaloTag>>> halo_full;  // (level, ng)
    DevBuf<PaFaceRec> face_recs;
    DevBuf<int> face_level;
    DevBuf<uint16_t> face_flags;
    DevBuf<PaFaceBlock> face_blocks;
    std::map<int, std::unique_ptr<DevBuf<long long>>> face_coff;   // coarse gather offsets per ghost width
    DevBuf<PaPackTag> pack_tags;
    TileTable tiles_simple, tiles_tma;
    // the same boxes cut into shallower work items (half / a quarter of the planes per item): picked at launch when the deepest
    // table would leave the persistent grid with only a handful of items per CTA (strong scaling: few boxes per rank)
    TileTable tiles_tma_fine[2];
    // ... and into deeper ones (four times the planes per item) for the flame-normal / divergence modes, which lose time at the
    // first plane of every item (the ring drains there) and gain 1.5-2 % from fewer, longer items where enough items remain
    TileTable tiles_tma_deep;
    // fused curvature (curv_fused.cu): K-block work items of every level (class 0 only) and the (level, box) list of the
    // shell pass; curv_ok = every local box is eligible (>= 3 cells in every direction, <= 128 wide, plane fits)
    TileTable tiles_curv;
    TileTable tiles_f3;                         // work items of the third fused kernel (curv_f3.cu): K rows x K planes x an x strip
    bool f3_ok = false;
    TileTable tiles_n3;                         // work items of its flame-normal-only form (PA_NORMAL_F3): rows x planes x strips of whole boxes
    bool n3_ok = false;
    TileTable tiles_nw;                         // work items of the barrier-free flame-normal kernel (normal_w.cu, PA_NORMAL_W)
    bool nw_ok = false;
    bool curv_ok = false;
    DevBuf<int> shell_level, shell_box;
    long long shell_begin[PA_MAX_LEVELS + 1] = {0};
    std::map<cudaStream_t, std::unique_ptr<DevBuf<double>>> staging;   // upload / download staging, one per stream
    std::map<cudaStream_t, std::unique_ptr<DevBuf<PaA4Dev>>> a4;       // per-box array records of device copies, one per stream
    DevBuf<double> send_slab, recv_slab;               // multi-rank exchange, [cell][comp]
    pa_field* recv_owner = nullptr;                    // the field whose exchanged data the (shared) recv slab holds right now
    int slab_ncomp = 0;
    // side stream on which the ghost fill of the refined levels overlaps the stencil of level 0 (created on demand)
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // filterPlt path: FillPatch tables per (level, ghost width, interpolater stencil), coarse-patch scratch, filter work prefix
    struct FpDev { DevBuf<PaFpPiece> pieces; DevBuf<PaFpCopy> copies; DevBuf<PaFpClamp> clamps; DevBuf<PaPackTag> pack; DevBuf<PaFpUnpack> unpack; };
    std::map<std::array<int, 3>, std::unique_ptr<FpDev>> fp;
    DevBuf<double> fp_scratch;
    // several ranks: slabs of the FillPatch exchange ([cell][comp], sized for the largest plan asked for) and the fill whose
    // data the recv slab holds right now (field, comp, ncomp, level, nghost, cgrow); any pack clears it
    DevBuf<double> fp_send, fp_recv;
    struct FpMark { const pa_field* f = nullptr; int comp = -1, ncomp = 0, lev = -1, ng = -1, cgrow = -1; } fp_mark;
    std::map<int, std::unique_ptr<DevBuf<long long>>> filter_prefix;   // per level
    std::map<int, long long> filter_nwork;
    DevBuf<double> filter_w3;
    // curvature temporaries (allocated on demand)
    pa_field* tmpG = nullptr;
    pa_field* tmpH = nullptr;
    pa_field* tmpW = nullptr;
    std::unique_ptr<SmoothDev> sm;
};

struct pa_field {
    pa_hier* h = nullptr;
    int ncomp = 0, ng = 0;
    std::vector<double*> slab;                         // per level
    std::vector<long long> cs;                         // component stride per level
    int recv_ncomp = 0;                                // >0: recv slab holds data for that many comps of this field
    int recv_comp0 = -1;
    // per level: where every rank's slab of this field lives (own allocation, or an IPC mapping of a peer's)
    std::vector<std::vector<PaPeerSlab>> peers_h;
    std::vector<std::unique_ptr<DevBuf<PaPeerSlab>>> peers_d;
    std::vector<void*> ipc_mapped;                     // pointers returned by cudaIpcOpenMemHandle
    int peers_missing = 0;                             // (level, rank) slabs with boxes that are not mapped yet
};

namespace {

const PaLayDev* dev_layout(pa_hier* h, int l, int ng, int* err) {
    auto key = std::make_pair(l, ng);
    auto it = h->lay.find(key);
    if (it != h->lay.end()) return it->second->p;
    const Layout& Y = h->H.layout(l, ng);
    auto buf = std::make_unique<DevBuf<PaLayDev>>();
    cudaError_t e = buf->upload(Y.lay, t_stream);
    if (e != cudaSuccess) { *err = cuda_fail(e, "upload layout"); return nullptr; }
    const PaLayDev* p = buf->p;
    h->lay.emplace(key, std::move(buf));
    return p;
}

void build_tiles(pa_hier* h, TileTable& T, bool tma, int zdiv = 1, int zmul = 1) {
    Hier& H = h->H;
    T.h.clear();
    T.max_plane_doubles = 0;
    T.ok = true;
    std::memset(T.begin, 0, sizeof(T.begin));
    std::memset(T.plane_doubles, 0, sizeof(T.plane_doubles));
    std::memset(T.items, 0, sizeof(T.items));
    const char* ety = getenv("PA_TMA_TY");
    const char* ezc = getenv("PA_TMA_ZC");
    const int TY0 = ety ? std::min(std::max(1, atoi(ety)), stencil_tma_max_tile_rows()) : stencil_tma_tile_rows();
    const int ZC0 = std::max(4, (ezc ? std::max(1, atoi(ezc)) : 32) * zmul / zdiv);
    for (int c = 0; c < (tma ? N_TILE_CLASSES : 1); ++c)
        for (int l = 0; l < H.nlev; ++l) {
            T.begin[c][l] = (long long)T.h.size();
            const Level& V = H.lev[l];
            const Layout& Y = H.layout(l, 1);
            for (size_t lb = 0; lb < V.local.size(); ++lb) {
                const Box& B = V.boxes[V.local[lb]];
                int nx = B.len(0), ny = B.len(1), nz = B.len(2);
                int ty, zc;
                if (tma) {
                    int nq = (nx + 1) / 2;
                    ty = std::min(TY0, std::max(1, 512 / nq));
                    if (nq > 512) T.ok = false;
                    // even split of the rows / planes so the last tile is not a sliver
                    int nty = (ny + ty - 1) / ty; ty = (ny + nty - 1) / nty;
                    int nzc = (nz + ZC0 - 1) / ZC0; zc = (nz + nzc - 1) / nzc;
                    const int it = nq * ty;
                    if (c != (it <= 128 ? 0 : it <= 256 ? 1 : 2)) continue;
                    const int plane = (ty + 2) * Y.lay[lb].P;
                    T.max_plane_doubles = std::max(T.max_plane_doubles, plane);
                    T.plane_doubles[c][l] = std::max(T.plane_doubles[c][l], plane);
                    T.items[c][l] = std::max(T.items[c][l], it);
                } else {
                    ty = 8; zc = 8;
                }
                for (int z0 = 0; z0 < nz; z0 += zc)
                    for (int y0 = 0; y0 < ny; y0 += ty) {
                        PaTile t;
                        t.lev = l; t.box = (int)lb;
                        t.y0 = y0; t.ny = std::min(ty, ny - y0);
                        t.z0 = z0; t.nz = std::min(zc, nz - z0);
                        T.h.push_back(t);
                    }
            }
            T.begin[c][l + 1] = (long long)T.h.size();
        }
    if (tma && T.max_plane_doubles > stencil_tma_max_plane_doubles()) T.ok = false;
}

// Work items of the fused curvature kernel: the K rows [1, ny-2] and K planes [1, nz-2] of every local box cut into blocks of
// at most (staged-row capacity - 4) rows and PA_CF_ZC planes; the kernel stages each block with a two-cell halo.  Items of one
// box are consecutive, y fastest, so neighbouring blocks -- which share halo rows -- are in flight at the same time and the
// re-read rows hit L2.
void build_curv_tiles(pa_hier* h, std::vector<int>& shell_level, std::vector<int>& shell_box) {
    Hier& H = h->H;
    TileTable& T = h->tiles_curv;
    T.h.clear();
    T.max_plane_doubles = 0;
    T.ok = true;
    std::memset(T.begin, 0, sizeof(T.begin));
    std::memset(T.plane_doubles, 0, sizeof(T.plane_doubles));
    std::memset(T.items, 0, sizeof(T.items));
    const char* ezc = getenv("PA_CF_ZC");
    const int ZC0 = ezc ? std::max(1, atoi(ezc)) : 64;
    const int cw = curv_fused_consumer_warps();
    shell_level.clear(); shell_box.clear();
    for (int l = 0; l < H.nlev; ++l) {
        T.begin[0][l] = (long long)T.h.size();
        h->shell_begin[l] = (long long)shell_level.size();
        const Level& V = H.lev[l];
        const Layout& Y = H.layout(l, 1);
        for (size_t lb = 0; lb < V.local.size(); ++lb) {
            const Box& B = V.boxes[V.local[lb]];
            const int nx = B.len(0), ny = B.len(1), nz = B.len(2);
            const int nq4 = (nx + 3) / 4;
            if (nx < 3 || ny < 3 || nz < 3 || nq4 > 32) { T.ok = false; continue; }
            int lpr = 1;
            while (lpr < nq4) lpr *= 2;
            // one n-row per LPR lanes of a consumer warp; the two halo rows of the staged block ride with the outermost n-rows
            const int rows_cap = std::min(cw * (32 / lpr) + 2, curv_fused_max_rows());
            int ty = rows_cap - 4;
            const int nky = ny - 2, nkz = nz - 2;
            const int nty = (nky + ty - 1) / ty; ty = (nky + nty - 1) / nty;
            const int nzc = (nkz + ZC0 - 1) / ZC0; const int zc = (nkz + nzc - 1) / nzc;
            const int plane = (ty + 4) * Y.lay[lb].P;
            T.max_plane_doubles = std::max(T.max_plane_doubles, plane);
            T.plane_doubles[0][l] = std::max(T.plane_doubles[0][l], plane);
            for (int z0 = 1; z0 < nz - 1; z0 += zc)
                for (int y0 = 1; y0 < ny - 1; y0 += ty) {
                    PaTile t;
                    t.lev = l; t.box = (int)lb;
                    t.y0 = y0; t.ny = std::min(ty, ny - 1 - y0);
                    t.z0 = z0; t.nz = std::min(zc, nz - 1 - z0);
                    T.h.push_back(t);
                }
            shell_level.push_back(l); shell_box.push_back((int)lb);
        }
        T.begin[0][l + 1] = (long long)T.h.size();
        h->shell_begin[l + 1] = (long long)shell_level.size();
    }
    if (T.max_plane_doubles > curv_fused_max_plane_doubles()) T.ok = false;
    h->curv_ok = T.ok;
    {   // third fused kernel: the same K rows / K planes cut into x strips of at most curv_f3_strip_pairs() pairs as well; the
        // strip (first pair, pairs) rides in the upper bits of PaTile::lev.  Strips of a row block are consecutive items.
        TileTable& F = h->tiles_f3;
        F.h.clear();
        F.ok = true;
        std::memset(F.begin, 0, sizeof(F.begin));
        const char* ez3 = getenv("PA_CF3_ZC");
        const int ZC3 = ez3 ? std::max(1, atoi(ez3)) : 63;
        const int ty3 = curv_f3_rows(), kq3 = curv_f3_strip_pairs();
        for (int l = 0; l < H.nlev; ++l) {
            F.begin[0][l] = (long long)F.h.size();
            const Level& V = H.lev[l];
            for (size_t lb = 0; lb < V.local.size(); ++lb) {
                const Box& B = V.boxes[V.local[lb]];
                const int nx = B.len(0), ny = B.len(1), nz = B.len(2);
                if (nx < 4 || (nx & 1) || nx > 256 || ny < 3 || nz < 3) { F.ok = false; continue; }
                const int nxp = nx / 2;
                const int nst = (nxp + kq3 - 1) / kq3, kq = (nxp + nst - 1) / nst;
                const int nky = ny - 2, nkz = nz - 2;
                const int nty = (nky + ty3 - 1) / ty3, ty = (nky + nty - 1) / nty;
                const int nzc = (nkz + ZC3 - 1) / ZC3, zc = (nkz + nzc - 1) / nzc;
                for (int z0 = 1; z0 < nz - 1; z0 += zc)
                    for (int y0 = 1; y0 < ny - 1; y0 += ty)
                        for (int q0 = 0; q0 < nxp; q0 += kq) {
                            PaTile t;
                            t.lev = l | (q0 << 8) | (std::min(kq, nxp - q0) << 16);
                            t.box = (int)lb;
                            t.y0 = y0; t.ny = std::min(ty, ny - 1 - y0);
                            t.z0 = z0; t.nz = std::min(zc, nz - 1 - z0);
                            F.h.push_back(t);
                        }
            }
            F.begin[0][l + 1] = (long long)F.h.size();
        }
        h->f3_ok = F.ok && !F.h.empty();
    }
    {   // the flame-normal-only form of that kernel: items tile the whole box (no rim), strips of at most normal_f3_strip_pairs() pairs
        TileTable& F = h->tiles_n3;
        F.h.clear();
        F.ok = true;
        std::memset(F.begin, 0, sizeof(F.begin));
        const char* ez = getenv("PA_NF3_ZC");
        const int ZC = ez ? std::max(1, atoi(ez)) : 64;
        const int ty0 = normal_f3_rows(), kq0 = normal_f3_strip_pairs();
        for (int l = 0; l < H.nlev; ++l) {
            F.begin[0][l] = (long long)F.h.size();
            const Level& V = H.lev[l];
            for (size_t lb = 0; lb < V.local.size(); ++lb) {
                const Box& B = V.boxes[V.local[lb]];
                const int nx = B.len(0), ny = B.len(1), nz = B.len(2);
                if (nx < 2 || (nx & 1) || nx > 510) { F.ok = false; continue; }
                const int nxp = nx / 2;
                const int nst = (nxp + kq0 - 1) / kq0, kq = (nxp + nst - 1) / nst;
                const int nty = (ny + ty0 - 1) / ty0, ty = (ny + nty - 1) / nty;
                const int nzc = (nz + ZC - 1) / ZC, zc = (nz + nzc - 1) / nzc;
                for (int z0 = 0; z0 < nz; z0 += zc)
                    for (int y0 = 0; y0 < ny; y0 += ty)
                        for (int q0 = 0; q0 < nxp; q0 += kq) {
                            PaTile t;
                            t.lev = l | (q0 << 8) | (std::min(kq, nxp - q0) << 16);
                            t.box = (int)lb;
                            t.y0 = y0; t.ny = std::min(ty, ny - y0);
                            t.z0 = z0; t.nz = std::min(zc, nz - z0);
                            F.h.push_back(t);
                        }
            }
            F.begin[0][l + 1] = (long long)F.h.size();
        }
        h->n3_ok = F.ok && !F.h.empty();
    }
    {   // normal_w.cu: one warp per row of an x strip of at most normal_w_strip_pairs() pairs (at least two), normal_w_rows() rows per item
        TileTable& F = h->tiles_nw;
        F.h.clear();
        F.ok = true;
        std::memset(F.begin, 0, sizeof(F.begin));
        const char* ez = getenv("PA_NW_ZC");
        const int ZC = ez ? std::max(1, atoi(ez)) : 32;
        const int ty0 = normal_w_rows(), kq0 = normal_w_strip_pairs();
        for (int l = 0; l < H.nlev; ++l) {
            F.begin[0][l] = (long long)F.h.size();
            const Level& V = H.lev[l];
            for (size_t lb = 0; lb < V.local.size(); ++lb) {
                const Box& B = V.boxes[V.local[lb]];
                const int nx = B.len(0), ny = B.len(1), nz = B.len(2);
                if (nx < 4 || (nx & 1) || nx > 510) { F.ok = false; continue; }
                const int nxp = nx / 2;
                const int nst = (nxp + kq0 - 1) / kq0, kq = (nxp + nst - 1) / nst;
                const int nzc = (nz + ZC - 1) / ZC, zc = (nz + nzc - 1) / nzc;
                for (int z0 = 0; z0 < nz; z0 += zc)
                    for (int y0 = 0; y0 < ny; y0 += ty0)
                        for (int q0 = 0; q0 < nxp; q0 += kq) {
                            PaTile t;
                            t.lev = l | (q0 << 8) | (std::min(kq, nxp - q0) << 16);
                            t.box = (int)lb;
                            t.y0 = y0; t.ny = std::min(ty0, ny - y0);
                            t.z0 = z0; t.nz = std::min(zc, nz - z0);
                            if ((t.lev >> 16) < 2) F.ok = false;
                            F.h.push_back(t);
                        }
            }
            F.begin[0][l + 1] = (long long)F.h.size();
        }
        h->nw_ok = F.ok && !F.h.empty();
    }
}

int ensure_device(pa_hier* h) {
    if (h->dev_ready) return PA_OK;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(PA_ERR_CUDA, std::string("no usable CUDA device (this library has no CPU fallback): ") + cudaGetErrorString(e));
    Hier& H = h->H;
    h->lev.clear();
    for (int l = 0; l < H.nlev; ++l) {
        auto D = std::make_unique<LevelDev>();
        const Level& V = H.lev[l];
        std::vector<PaBoxDev> bd;
        D->host_off_h.assign(1, 0);
        for (size_t e = 0; e < V.ext.size(); ++e) {
            const int gb = V.ext[e];
            PaBoxDev b;
            for (int d = 0; d < 3; ++d) { b.lo[d] = V.boxes[gb].lo[d]; b.n[d] = V.boxes[gb].len(d); }
            bd.push_back(b);
            if (e < V.local.size()) D->host_off_h.push_back(D->host_off_h.back() + V.boxes[gb].npts());
        }
        CU(D->boxes.upload(bd, t_stream));
        CU(D->nbr.upload(V.nbr, t_stream));
        CU(D->halo_cross.upload(H.halo_cross[l].tags, t_stream));
        CU(D->host_off.upload(D->host_off_h, t_stream));
        CU(D->gid.upload(V.local, t_stream));
        h->lev.push_back(std::move(D));
    }
    CU(h->face_recs.upload(H.faces.recs, t_stream));
    CU(h->face_level.upload(H.faces.rec_level, t_stream));
    CU(h->face_flags.upload(H.faces.flags, t_stream));
    CU(h->face_blocks.upload(H.faces.blocks, t_stream));
    CU(h->pack_tags.upload(H.xplan.pack, t_stream));
    build_tiles(h, h->tiles_simple, false);
    build_tiles(h, h->tiles_tma, true);
    CU(h->tiles_simple.d.upload(h->tiles_simple.h, t_stream));
    CU(h->tiles_tma.d.upload(h->tiles_tma.h, t_stream));
    for (int k = 0; k < 2; ++k) {
        build_tiles(h, h->tiles_tma_fine[k], true, 2 << k);
        CU(h->tiles_tma_fine[k].d.upload(h->tiles_tma_fine[k].h, t_stream));
    }
    build_tiles(h, h->tiles_tma_deep, true, 1, 4);
    CU(h->tiles_tma_deep.d.upload(h->tiles_tma_deep.h, t_stream));
    {
        std::vector<int> sl, sb;
        build_curv_tiles(h, sl, sb);
        if (h->f3_ok) CU(h->tiles_f3.d.upload(h->tiles_f3.h, t_stream));
        if (h->n3_ok) CU(h->tiles_n3.d.upload(h->tiles_n3.h, t_stream));
        if (h->nw_ok) CU(h->tiles_nw.d.upload(h->tiles_nw.h, t_stream));
        if (h->curv_ok) {
            CU(h->tiles_curv.d.upload(h->tiles_curv.h, t_stream));
            CU(h->shell_level.upload(sl, t_stream));
            CU(h->shell_box.upload(sb, t_stream));
            CU(cudaStreamSynchronize(t_stream));   // sl / sb die at the end of this scope
        }
    }
    CU(cudaStreamSynchronize(t_stream));      // host vectors may be reallocated later
    h->dev_ready = true;
    return PA_OK;
}

int ensure_slabs(pa_hier* h, int ncomp) {
    Hier& H = h->H;
    if (H.nranks <= 1) return PA_OK;
    size_t ns = (size_t)H.xplan.send_prefix[H.nranks] * ncomp, nr = (size_t)H.xplan.recv_prefix[H.nranks] * ncomp;
    CU(h->send_slab.reserve(std::max<size_t>(ns, 1)));
    CU(h->recv_slab.reserve(std::max<size_t>(nr, 1)));
    return PA_OK;
}

// GridArgs with `in` = `out` = comp `comp` of field f (in-place operations: ghost fill, pack)
int grid_args_inplace(pa_field* f, int comp, GridArgs& ga) {
    pa_hier* h = f->h;
    std::memset(&ga, 0, sizeof(ga));
    for (int l = 0; l < h->H.nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* ly = dev_layout(h, l, f->ng, &err);
        if (!ly && !h->H.lev[l].local.empty()) return err;
        LevArgs& A = ga.L[l];
        A.boxes = h->lev[l]->boxes.p;
        A.lay_in = A.lay_out = ly;
        A.nbr = h->lev[l]->nbr.p;
        A.peers = f->peers_d[l]->p;
        A.in_comp = comp;
        A.in = A.out = f->slab[l] ? f->slab[l] + (long long)comp * f->cs[l] : nullptr;
        A.cs_in = A.cs_out = f->cs[l];
        for (int d = 0; d < 3; ++d) A.dxi[d] = h->H.lev[l].dxinv[d];
    }
    return PA_OK;
}

int grid_args(pa_field* in, int comp_in, pa_field* out, int comp_out, GridArgs& ga) {
    pa_hier* h = in->h;
    std::memset(&ga, 0, sizeof(ga));
    for (int l = 0; l < h->H.nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* li = dev_layout(h, l, in->ng, &err);
        if (!li && !h->H.lev[l].local.empty()) return err;
        const PaLayDev* lo = dev_layout(h, l, out->ng, &err);
        if (!lo && !h->H.lev[l].local.empty()) return err;
        LevArgs& A = ga.L[l];
        A.boxes = h->lev[l]->boxes.p;
        A.lay_in = li; A.lay_out = lo;
        A.nbr = h->lev[l]->nbr.p;
        A.peers = in->peers_d[l]->p;
        A.in_comp = comp_in;
        A.in = in->slab[l] ? in->slab[l] + (long long)comp_in * in->cs[l] : nullptr;
        A.out = out->slab[l] ? out->slab[l] + (long long)comp_out * out->cs[l] : nullptr;
        A.cs_in = in->cs[l]; A.cs_out = out->cs[l];
        for (int d = 0; d < 3; ++d) A.dxi[d] = h->H.lev[l].dxinv[d];
    }
    return PA_OK;
}

bool use_tma(pa_hier* h, int nin) {
    const char* e = getenv("PA_STENCIL");
    if (e && !strcmp(e, "simple")) return false;
    if (!h->tiles_tma.ok) return false;
    // shared memory: STAGES(4) * nin * stage_doubles * 8 bytes must fit in 227 KB
    long long stage = (h->tiles_tma.max_plane_doubles + 15) & ~15;
    return 4LL * nin * stage * 8 <= 200 * 1024;
}

// stencil over levels [l0, l1]
int run_stencil(pa_hier* h, int mode, const GridArgs& ga, const StencilExtra& ex, int nvar, int l0, int l1, int in_ng,
                const pa_field* in) {
    const int nin = (mode == MODE_DIV) ? 3 : 1;
    if (mode == MODE_NORMAL_S && !(in_ng == 1 && use_tma(h, 1))) return fail(PA_ERR_STATE, "internal: MODE_NORMAL_S needs the TMA pipeline");
    if (in->peers_missing > 0)
        return fail(PA_ERR_STATE, "this hierarchy uses peer links (PA_HIER_PEER_LINKS): map every rank's slab of the input field first "
                                  "(pa_field_ipc_handle -> exchange -> pa_field_map_peer)");
    // the TMA tile table is sized for the nghost == 1 layout (row pitch nx+4)
    if (in_ng == 1 && use_tma(h, nin)) {
        // Work items per launch: (tiles of the level range) x variables, drawn dynamically by 148 x 2 (or so) persistent CTAs.
        // With few items per CTA the last round of items leaves most SMs idle (strong scaling at 8 ranks): take the table
        // with half / a quarter of the planes per item then.  Measured on the per-rank load of configs[1] at N = 8 (8 boxes x 5
        // variables, 8.65 items per slot): 93.1 / 95.7 / 97.0 % of the HBM roofline for 32 / 16 / 8 planes per item
        // (profiles/r02_ab_zdiv.txt) -- the bandwidth-bound gradient modes switch below 24 items per slot.  The flame-normal
        // and divergence modes pay more per item (first-plane wait of a deeper ring) and were 3-5 % slower with shallower
        // items on large workloads: they switch only below 8.  PA_TMA_ZDIV=0|1|2 forces one.
        TileTable* Tp = &h->tiles_tma;
        {
            cudaError_t esm = cudaSuccess;
            const long long slots = 2LL * std::max(1, stencil_num_sms(&esm));
            const char* ez = getenv("PA_TMA_ZDIV");
            int pick = 0;
            if (ez) pick = std::min(2, std::max(0, atoi(ez)));
            else {
                auto items = [&](const TileTable& X) { long long n = 0; for (int c = 0; c < N_TILE_CLASSES; ++c) n += X.begin[c][l1 + 1] - X.begin[c][l0]; return n * nvar; };
                const long long want = (mode == MODE_GRAD || mode == MODE_GRAD3) ? 24 : 8;
                while (pick < 2 && items(pick == 0 ? h->tiles_tma : h->tiles_tma_fine[pick - 1]) < want * slots) ++pick;
            }
            if (pick > 0 && h->tiles_tma_fine[pick - 1].ok) Tp = &h->tiles_tma_fine[pick - 1];
            // measured (profiles/r02_ab_zc_curvature.txt): 128 instead of 32 planes per item, curvature on the north-star
            // hierarchy 6.66 -> 6.53 ms; on 64^3 boxes (5 items per slot left) 1.024 -> 1.034 ms, hence the item-count condition
            const bool heavy = mode == MODE_NORMAL || mode == MODE_NORMAL_S || mode == MODE_DIV;
            if (!ez && pick == 0 && heavy && h->tiles_tma_deep.ok) {
                long long n = 0;
                for (int c = 0; c < N_TILE_CLASSES; ++c) n += h->tiles_tma_deep.begin[c][l1 + 1] - h->tiles_tma_deep.begin[c][l0];
                if (n * nvar >= 8 * slots) Tp = &h->tiles_tma_deep;
            }
        }
        TileTable& T = *Tp;
        for (int c = 0; c < N_TILE_CLASSES; ++c) {
            const long long a = T.begin[c][l0], b = T.begin[c][l1 + 1];
            if (b <= a) continue;
            // stage size and CTA shape follow the largest tile of this class on the levels of the launch
            int plane = 0, items = 0;
            for (int l = l0; l <= l1; ++l) { plane = std::max(plane, T.plane_doubles[c][l]); items = std::max(items, T.items[c][l]); }
            CU(launch_stencil_tma(mode, T.d.p + a, (int)(b - a), plane, items, ga, ex, nvar, t_stream));
        }
    } else {
        TileTable& T = h->tiles_simple;
        long long a = T.begin[0][l0], b = T.begin[0][l1 + 1];
        CU(launch_stencil_simple(mode, T.d.p + a, (int)(b - a), ga, ex, nvar, t_stream));
    }
    return PA_OK;
}

int check_field(const pa_field* f, int comp, int ncomp, const char* who) {
    if (!f || !f->h) return fail(PA_ERR_ARG, std::string(who) + ": null field");
    if (comp < 0 || ncomp < 1 || comp + ncomp > f->ncomp) return fail(PA_ERR_ARG, std::string(who) + ": component range out of bounds");
    return PA_OK;
}

// ghost fill of comps [comp, comp+ncomp) on levels [l0, l1]: halo gather per level + one BC-fill launch.
// linked_too = false (the product path): faces with a neighbour link are skipped -- the stencil kernels read the
// neighbour in place; true: every ghost cell of the width-1 face layers is materialised (pa_fill_ghosts).
// recs: face records to use instead of the hierarchy's (pa_smooth's coarse-fine polynomial order); same order and extents.
int fill_ghosts_impl(pa_field* f, int comp, int ncomp, int l0, int l1, bool linked_too, GhostXform xf = GhostXform{0, 0.0, 1.0},
                     const PaFaceRec* recs = nullptr) {
    pa_hier* h = f->h;
    Hier& H = h->H;
    CHK(ensure_device(h));
    if (f->ng < 1) return fail(PA_ERR_ARG, "ghost fill needs a field with nghost >= 1");
    if (H.filter_only)
        return fail(PA_ERR_UNSUPPORTED, "this hierarchy was created with PA_HIER_FILTER_ONLY: it has no coarse-fine / wall face tables; "
                                        "grad, curvature and pa_fill_ghosts need a hierarchy created without that flag");
    const double* recv = nullptr;
    if (H.nranks > 1 && H.xplan.recv_prefix[H.nranks] + H.xplan.send_prefix[H.nranks] > 0) {
        if (f->recv_ncomp != ncomp || f->recv_comp0 != comp)
            return fail(PA_ERR_STATE, "multi-rank ghost fill: exchange this component range first (pa_exchange_pack -> transport -> pa_exchange_mark_received)");
        recv = h->recv_slab.p;
    }
    // with peer links the coarse cells of coarse-fine faces owned by other ranks are read in place, as linked faces are
    if ((linked_too || (H.peer_links && H.nranks > 1 && H.nlev > 1)) && f->peers_missing > 0)
        return fail(PA_ERR_STATE, "peer links: map every rank's slab of this field first (pa_field_map_peer)");
    GridArgs ga;
    CHK(grid_args_inplace(f, comp, ga));
    for (int l = l0; l <= l1; ++l) {
        const HaloTable& T = H.halo_cross[l];
        const int t1 = linked_too ? (int)T.tags.size() : T.ntags_unlinked;
        const long long c1 = linked_too ? T.ncells : T.ncells_unlinked;
        CU(launch_halo(h->lev[l]->halo_cross.p, 0, t1, 0, c1, ga.L[l].boxes, ga.L[l].lay_in, ga.L[l].out,
                       f->cs[l], ncomp, recv, ga.L[l].peers, comp, H.rank, xf, t_stream));
    }
    const FaceTable& F = H.faces;
    const long long b0 = F.level_blk_begin[l0], b1 = F.level_blk_begin[l1 + 1];
    if (b1 > b0) {
        auto it = h->face_coff.find(f->ng);
        if (it == h->face_coff.end()) {
            auto buf = std::make_unique<DevBuf<long long>>();
            std::vector<long long> v = H.crse_offsets(f->ng);
            CU(buf->upload(v, t_stream));
            CU(cudaStreamSynchronize(t_stream));           // v dies at the end of this scope
            it = h->face_coff.emplace(f->ng, std::move(buf)).first;
        }
        CU(launch_bcfill(recs ? recs : h->face_recs.p, h->face_level.p, h->face_blocks.p, b0, b1, h->face_flags.p, it->second->p, ga, ncomp, recv, xf, t_stream));
    }
    return PA_OK;
}

// ---- overlap of the refined levels' ghost fill with the stencil of level 0 -----------------------------------------
// The BC fill of levels >= 1 is a latency-bound gather (coarse VALID cells + fine interior cells -> fine ghost cells) that
// depends on nothing the level-0 stencil writes, and level 0 is a third or more of the cells of a hierarchy.  So one pass is
//     caller's stream:  fill(level 0)  | stencil(level 0)            | wait | stencil(levels >= 1)
//     side stream:      wait(fork)     | fill(levels >= 1)  record   |
// Opt-in (PA_STREAM_OVERLAP=1).  Measured on B200 it does NOT pay (profiles/r01_ab_stream_overlap.txt: curvature on the
// target hierarchy 6.90 ms with it, 6.59 ms without; grad on 16^3 boxes 0.997 vs 0.983 ms): the persistent stencil kernels
// own the SMs, so the fill's blocks mostly wait anyway, and splitting each stencil pass in two costs a second ramp-up and
// tail.  The default therefore keeps everything on the caller's stream in the plain order fill(all) -> stencil(all).
bool overlap_enabled(const pa_hier* h) {
    if (h->H.nlev < 2) return false;
    const char* e = getenv("PA_STREAM_OVERLAP");
    return e && e[0] == '1';
}
int ensure_side(pa_hier* h) {
    if (h->side) return PA_OK;
    CU(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    return PA_OK;
}
// run `fill_fine` (a ghost fill of levels >= 1) on the side stream, ordered after everything already enqueued on the
// caller's stream; the caller's stream goes on and must call join_side() before it touches what the fill wrote
template <class F>
int fork_side(pa_hier* h, F&& fill_fine) {
    CHK(ensure_side(h));
    cudaStream_t main_stream = t_stream;
    CU(cudaEventRecord(h->ev_fork, main_stream));
    CU(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
    t_stream = h->side;
    const int rc = fill_fine();
    t_stream = main_stream;
    CHK(rc);
    CU(cudaEventRecord(h->ev_join, h->side));
    return PA_OK;
}
int join_side(pa_hier* h) {
    CU(cudaStreamWaitEvent(t_stream, h->ev_join, 0));
    return PA_OK;
}

// the multigrid preconditioner's fields and level-0 coarsenings (fields before the hierarchies they live on)
void free_smooth_mg(SmoothDev& S) {
    for (auto& f : S.mg_f) for (pa_field* g : f) if (g) pa_field_free(g);
    for (pa_hier* m : S.mg_h) pa_hier_destroy(m);
    if (S.mg_rhs) pa_field_free(S.mg_rhs);
    if (S.mg_res) pa_field_free(S.mg_res);
    S.mg_f.clear();
    S.mg_h.clear();
    S.mg_rhs = S.mg_res = nullptr;
    S.mg_ready = false;
}

}  // namespace

// =============================================================================================================
extern "C" {

const char* pa_last_error(void) { return t_err.c_str(); }
const char* pa_version(void) { return "pele-stencil-b200 0.1 (sm_100a)"; }

int pa_init(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(PA_ERR_CUDA, std::string("pa_init: no usable CUDA device (no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(PA_ERR_ARG, "pa_init: device index out of range");
    CU(cudaSetDevice(device));
    cudaDeviceProp p;
    CU(cudaGetDeviceProperties(&p, device));
    if (p.major < 10) return fail(PA_ERR_UNSUPPORTED, "pa_init: kernels are built for sm_100a only; device is sm_" + std::to_string(p.major) + std::to_string(p.minor));
    return PA_OK;
}
int pa_finalize(void) { stencil_tma_release(); return PA_OK; }
int pa_set_stream(void* s) { t_stream = (cudaStream_t)s; return PA_OK; }
int pa_sync(void) { CU(cudaStreamSynchronize(t_stream)); return PA_OK; }
int pa_host_alloc(void** p, size_t bytes) { CU(cudaHostAlloc(p, bytes, cudaHostAllocDefault)); return PA_OK; }
int pa_host_free(void* p) { CU(cudaFreeHost(p)); return PA_OK; }
int pa_host_register(void* p, size_t bytes) { CU(cudaHostRegister(p, bytes, cudaHostRegisterDefault)); return PA_OK; }
int pa_host_unregister(void* p) { CU(cudaHostUnregister(p)); return PA_OK; }
int64_t pa_kernel_launches(void) { return g_launches; }
int pa_debug_device_bytes(int64_t* out) {
    if (!out) return fail(PA_ERR_ARG, "pa_debug_device_bytes: null output");
    int dev = 0;
    CU(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_alloc_mu);
    auto it = g_alloc_bytes.find(dev);
    *out = it == g_alloc_bytes.end() ? 0 : it->second;
    return PA_OK;
}

int pa_hier_create(pa_hier** out, int nlev, const pa_level_desc* levels, const int is_per[3], const int bc_kind[3],
                   int rank, int nranks) {
    return pa_hier_create2(out, nlev, levels, is_per, bc_kind, rank, nranks, 0u);
}

int pa_hier_create2(pa_hier** out, int nlev, const pa_level_desc* levels, const int is_per[3], const int bc_kind[3],
                    int rank, int nranks, unsigned flags) {
    if (flags & ~(unsigned)(PA_HIER_PEER_LINKS | PA_HIER_NO_LINKS | PA_HIER_FILTER_ONLY)) return fail(PA_ERR_ARG, "pa_hier_create2: unknown flag");
    if (!out || !levels || !is_per) return fail(PA_ERR_ARG, "pa_hier_create: null argument");
    std::vector<pa_level_desc_host> L(std::max(nlev, 0));
    for (int l = 0; l < nlev; ++l) {
        for (int d = 0; d < 3; ++d) {
            L[l].domain_lo[d] = levels[l].domain_lo[d]; L[l].domain_hi[d] = levels[l].domain_hi[d];
            L[l].dx[d] = levels[l].dx[d];
        }
        L[l].nboxes = levels[l].nboxes; L[l].boxes = levels[l].boxes; L[l].owner = levels[l].owner;
        if (!L[l].boxes) return fail(PA_ERR_ARG, "pa_hier_create: level without boxes");
    }
    auto h = std::make_unique<pa_hier>();
    std::string e = h->H.init(nlev, L.data(), is_per, bc_kind, rank, nranks, flags);
    if (!e.empty()) return fail(PA_ERR_ARG, "pa_hier_create: " + e);
    *out = h.release();
    return PA_OK;
}

int pa_hier_destroy(pa_hier* h) {
    if (!h) return PA_OK;
    if (h->tmpG) pa_field_free(h->tmpG);
    if (h->tmpH) pa_field_free(h->tmpH);
    if (h->tmpW) pa_field_free(h->tmpW);
    if (h->sm) {
        for (pa_field* f : h->sm->w) if (f) pa_field_free(f);
        free_smooth_mg(*h->sm);
    }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->side) cudaStreamDestroy(h->side);
    delete h;
    return PA_OK;
}
int pa_hier_num_levels(const pa_hier* h) { return h ? h->H.nlev : 0; }
int pa_hier_num_boxes(const pa_hier* h, int lev) { return (h && lev >= 0 && lev < h->H.nlev) ? (int)h->H.lev[lev].boxes.size() : -1; }
int64_t pa_hier_num_cells(const pa_hier* h, int lev) {
    if (!h) return 0;
    if (lev >= 0) return lev < h->H.nlev ? h->H.lev[lev].ncells : 0;
    int64_t s = 0;
    for (auto& l : h->H.lev) s += l.ncells;
    return s;
}
int64_t pa_hier_num_local_cells(const pa_hier* h, int lev) {
    if (!h) return 0;
    if (lev >= 0) return lev < h->H.nlev ? h->H.lev[lev].ncells_local : 0;
    int64_t s = 0;
    for (auto& l : h->H.lev) s += l.ncells_local;
    return s;
}
int pa_hier_box_owner(const pa_hier* h, int lev, int box) {
    if (!h || lev < 0 || lev >= h->H.nlev || box < 0 || box >= (int)h->H.lev[lev].boxes.size()) return -1;
    return h->H.lev[lev].owner[box];
}
int pa_hier_build_seconds(const pa_hier* h, double* s) { if (!h || !s) return fail(PA_ERR_ARG, "null"); *s = h->H.build_seconds; return PA_OK; }

int pa_sfc_distribute(int nboxes, const int* boxes, int nranks, int* owner_out) {
    if (nboxes < 1 || !boxes || nranks < 1 || !owner_out) return fail(PA_ERR_ARG, "pa_sfc_distribute: bad argument");
    sfc_distribute(nboxes, boxes, nranks, owner_out);
    return PA_OK;
}

int64_t pa_algorithmic_bytes(const pa_hier* h, int nout) {
    if (!h) return 0;
    int64_t s = 0;
    for (auto& V : h->H.lev)
        for (int gb : V.local) {
            const Box& B = V.boxes[gb];
            int64_t nx = B.len(0), ny = B.len(1), nz = B.len(2);
            int64_t vol = nx * ny * nz;
            s += 8 * (vol + 2 * (nx * ny + ny * nz + nx * nz)) + 8 * (int64_t)nout * vol;
        }
    return s;
}

// ---------------------------------------------------------------------------------------------- fields
int pa_field_alloc(pa_hier* h, int ncomp, int nghost, pa_field** out) {
    if (!h || !out || ncomp < 1 || nghost < 0 || nghost > 32) return fail(PA_ERR_ARG, "pa_field_alloc: bad argument (ncomp >= 1, 0 <= nghost <= 32)");
    CHK(ensure_device(h));
    auto f = std::make_unique<pa_field>();
    f->h = h; f->ncomp = ncomp; f->ng = nghost;
    f->slab.assign(h->H.nlev, nullptr);
    f->cs.assign(h->H.nlev, 0);
    f->peers_h.assign(h->H.nlev, std::vector<PaPeerSlab>(h->H.nranks, PaPeerSlab{nullptr, 0}));
    for (int l = 0; l < h->H.nlev; ++l) f->peers_d.push_back(std::make_unique<DevBuf<PaPeerSlab>>());
    for (int l = 0; l < h->H.nlev; ++l) {
        const Layout& Y = h->H.layout(l, nghost);
        f->cs[l] = Y.comp_stride;
        for (int r = 0; r < h->H.nranks; ++r) {
            f->peers_h[l][r].cs = Y.rank_comp_stride[r];
            if (r != h->H.rank && h->H.peer_links && Y.rank_comp_stride[r] > 0) ++f->peers_missing;
        }
        size_t n = (size_t)Y.comp_stride * ncomp + 16;          // 16 doubles of slack: pair loads may touch one element past a row
        if (Y.comp_stride == 0) continue;
        cudaError_t e = dev_alloc((void**)&f->slab[l], n * sizeof(double));
        if (e != cudaSuccess) {
            for (double* p : f->slab) if (p) dev_free(p);
            return e == cudaErrorMemoryAllocation ? fail(PA_ERR_NOMEM, "pa_field_alloc: out of device memory") : cuda_fail(e, "cudaMalloc");
        }
        // ghost cells and pads start as zeros (never NaN garbage)
        CU(cudaMemsetAsync(f->slab[l], 0, n * sizeof(double), t_stream));
        int err = PA_OK;
        if (!dev_layout(h, l, nghost, &err)) return err;
    }
    for (int l = 0; l < h->H.nlev; ++l) {
        f->peers_h[l][h->H.rank].base = f->slab[l];
        CU(f->peers_d[l]->upload(f->peers_h[l], t_stream));
    }
    CU(cudaStreamSynchronize(t_stream));               // peers_h may be modified by pa_field_map_peer
    *out = f.release();
    return PA_OK;
}
int pa_field_free(pa_field* f) {
    if (!f) return PA_OK;
    if (f->h && f->h->recv_owner == f) f->h->recv_owner = nullptr;
    if (f->h && f->h->fp_mark.f == f) f->h->fp_mark = pa_hier::FpMark();
    for (void* p : f->ipc_mapped) cudaIpcCloseMemHandle(p);
    for (double* p : f->slab) if (p) dev_free(p);
    delete f;
    return PA_OK;
}
int pa_field_ncomp(const pa_field* f) { return f ? f->ncomp : -1; }
int pa_field_nghost(const pa_field* f) { return f ? f->ng : -1; }
int64_t pa_field_bytes(const pa_field* f) {
    if (!f) return 0;
    int64_t s = 0;
    for (size_t l = 0; l < f->cs.size(); ++l) s += (int64_t)f->cs[l] * f->ncomp * 8;
    return s;
}

// ---- peer mapping (one process per GPU; CUDA IPC over NVLink) --------------------------------------------------
int pa_field_ipc_handle(const pa_field* f, int lev, void* handle64) {
    if (!f || !handle64 || lev < 0 || lev >= f->h->H.nlev) return fail(PA_ERR_ARG, "pa_field_ipc_handle: bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    std::memset(handle64, 0, 64);
    if (!f->slab[lev]) return PA_OK;                   // this rank owns no box of the level
    cudaIpcMemHandle_t hd;
    CU(cudaIpcGetMemHandle(&hd, f->slab[lev]));
    std::memcpy(handle64, &hd, 64);
    return PA_OK;
}

static int set_peer_base(pa_field* f, int lev, int peer_rank, const double* base) {
    pa_hier* h = f->h;
    f->peers_h[lev][peer_rank].base = base;
    CU(f->peers_d[lev]->upload(f->peers_h[lev], t_stream));
    CU(cudaStreamSynchronize(t_stream));
    if (h->H.peer_links && f->peers_missing > 0) --f->peers_missing;
    return PA_OK;
}

int pa_field_map_peer(pa_field* f, int lev, int peer_rank, const void* handle64) {
    if (!f || !handle64 || lev < 0 || lev >= f->h->H.nlev || peer_rank < 0 || peer_rank >= f->h->H.nranks)
        return fail(PA_ERR_ARG, "pa_field_map_peer: bad argument");
    pa_hier* h = f->h;
    if (peer_rank == h->H.rank) return PA_OK;
    PaPeerSlab& S = f->peers_h[lev][peer_rank];
    if (S.cs == 0) return PA_OK;                       // the peer owns no box of this level
    if (S.base) return fail(PA_ERR_STATE, "pa_field_map_peer: this (level, rank) is already mapped");
    cudaIpcMemHandle_t hd;
    std::memcpy(&hd, handle64, 64);
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
    f->ipc_mapped.push_back(p);
    return set_peer_base(f, lev, peer_rank, (const double*)p);
}

// ---- the same for ranks that live in ONE process (one host thread per GPU): no IPC, the peer's pointer is valid here --
int pa_enable_peer_access(int peer_device) {
    cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return PA_OK; }
    if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
    return PA_OK;
}
int pa_field_slab(const pa_field* f, int lev, const double** base) {
    if (!f || !base || lev < 0 || lev >= f->h->H.nlev) return fail(PA_ERR_ARG, "pa_field_slab: bad argument");
    *base = f->slab[lev];
    return PA_OK;
}
int pa_field_map_peer_ptr(pa_field* f, int lev, int peer_rank, const double* base) {
    if (!f || lev < 0 || lev >= f->h->H.nlev || peer_rank < 0 || peer_rank >= f->h->H.nranks)
        return fail(PA_ERR_ARG, "pa_field_map_peer_ptr: bad argument");
    if (peer_rank == f->h->H.rank) return PA_OK;
    PaPeerSlab& S = f->peers_h[lev][peer_rank];
    if (S.cs == 0) return PA_OK;                       // the peer owns no box of this level
    if (!base) return fail(PA_ERR_ARG, "pa_field_map_peer_ptr: the peer owns boxes of this level but gave no slab");
    if (S.base) return fail(PA_ERR_STATE, "pa_field_map_peer_ptr: this (level, rank) is already mapped");
    return set_peer_base(f, lev, peer_rank, base);
}
int pa_copy_async(double* dst, const double* src, int64_t n) {
    if (n <= 0) return PA_OK;
    if (!dst || !src) return fail(PA_ERR_ARG, "pa_copy_async: null pointer");
    CU(cudaMemcpyAsync(dst, src, (size_t)n * sizeof(double), cudaMemcpyDefault, t_stream));
    return PA_OK;
}

static int box_copy(const pa_field* f, int lev, int box, int comp, double* host, bool to_dev, bool grown) {
    if (!f) return fail(PA_ERR_ARG, "null field");
    pa_hier* h = f->h;
    if (lev < 0 || lev >= h->H.nlev || comp < 0 || comp >= f->ncomp) return fail(PA_ERR_ARG, "level / component out of range");
    const Level& V = h->H.lev[lev];
    if (box < 0 || box >= (int)V.boxes.size()) return fail(PA_ERR_ARG, "box out of range");
    int lb = V.g2l[box];
    if (lb < 0) return fail(PA_ERR_ARG, "box is owned by another rank");
    const Box& B = V.boxes[box];
    const PaLayDev& y = h->H.layout(lev, f->ng).lay[lb];
    const int g = grown ? f->ng : 0;
    const int nx = B.len(0) + 2 * g, ny = B.len(1) + 2 * g, nz = B.len(2) + 2 * g;
    double* base = f->slab[lev] + (long long)comp * f->cs[lev] + y.off + (long long)(y.ng - g) * y.PS + (long long)(y.ng - g) * y.P + (y.ng - g + y.xoff);
    // plane by plane 2-D copies: device rows have pitch P, planes PS (not a multiple of the row count of the sub-box)
    for (int k = 0; k < nz; ++k) {
        double* dp = base + (long long)k * y.PS;
        double* hp = host + (long long)k * nx * ny;
        if (to_dev) CU(cudaMemcpy2DAsync(dp, (size_t)y.P * 8, hp, (size_t)nx * 8, (size_t)nx * 8, ny, cudaMemcpyHostToDevice, t_stream));
        else CU(cudaMemcpy2DAsync(hp, (size_t)nx * 8, dp, (size_t)y.P * 8, (size_t)nx * 8, ny, cudaMemcpyDeviceToHost, t_stream));
    }
    return PA_OK;
}
int pa_field_upload(pa_field* f, int lev, int box, int comp, const double* host) {
    return box_copy(f, lev, box, comp, const_cast<double*>(host), true, false);
}
int pa_field_download(const pa_field* f, int lev, int box, int comp, double* host) {
    return box_copy(f, lev, box, comp, host, false, false);
}
int pa_debug_download_grown(const pa_field* f, int lev, int box, int comp, double* host) {
    CHK(box_copy(f, lev, box, comp, host, false, true));
    CU(cudaStreamSynchronize(t_stream));
    return PA_OK;
}

// Whole-level transfers.  Boxes with rows of >= 512 bytes go box by box as pitched 3-D DMA copies straight between the
// caller's (pinned) buffer and the padded device layout: no staging buffer, no kernel, nothing shared between streams,
// so uploads, compute and downloads of different components can overlap on different streams.  Levels made of small
// boxes (short rows are slow for the copy engines) take one contiguous copy through a per-stream staging buffer plus one
// pack / unpack kernel.
static bool level_uses_dma(const pa_hier* h, int lev) {
    const Level& V = h->H.lev[lev];
    for (int gb : V.local) if (V.boxes[gb].len(0) * 8 < 512) return false;
    return true;
}

static int level_dma(const pa_field* f, int lev, int comp, double* host, bool to_dev) {
    pa_hier* h = f->h;
    const Level& V = h->H.lev[lev];
    const Layout& Y = h->H.layout(lev, f->ng);
    long long ho = 0;
    for (size_t lb = 0; lb < V.local.size(); ++lb) {
        const Box& B = V.boxes[V.local[lb]];
        const PaLayDev& y = Y.lay[lb];
        const size_t nx = B.len(0), ny = B.len(1), nz = B.len(2);
        cudaMemcpy3DParms p;
        std::memset(&p, 0, sizeof(p));
        cudaPitchedPtr hp = make_cudaPitchedPtr(host + ho, nx * 8, nx * 8, ny);
        cudaPitchedPtr dp = make_cudaPitchedPtr(f->slab[lev] + (long long)comp * f->cs[lev] + y.off, (size_t)y.P * 8, (size_t)y.P * 8, (size_t)(y.PS / y.P));
        cudaPos dpos = make_cudaPos((size_t)(y.ng + y.xoff) * 8, (size_t)y.ng, (size_t)y.ng);
        if (to_dev) { p.srcPtr = hp; p.dstPtr = dp; p.dstPos = dpos; p.kind = cudaMemcpyHostToDevice; }
        else { p.srcPtr = dp; p.srcPos = dpos; p.dstPtr = hp; p.kind = cudaMemcpyDeviceToHost; }
        p.extent = make_cudaExtent(nx * 8, ny, nz);
        CU(cudaMemcpy3DAsync(&p, t_stream));
        ho += (long long)B.npts();
    }
    return PA_OK;
}

static int stream_staging(pa_hier* h, size_t n, double** out) {
    auto& slot = h->staging[t_stream];
    if (!slot) slot = std::make_unique<DevBuf<double>>();
    CU(slot->reserve(n));
    *out = slot->p;
    return PA_OK;
}

int pa_field_upload_level(pa_field* f, int lev, int comp, const double* host) {
    if (!f || lev < 0 || lev >= f->h->H.nlev || comp < 0 || comp >= f->ncomp || !host) return fail(PA_ERR_ARG, "pa_field_upload_level: bad argument");
    pa_hier* h = f->h;
    LevelDev& D = *h->lev[lev];
    long long n = D.host_off_h.back();
    if (n == 0) return PA_OK;
    if (level_uses_dma(h, lev)) return level_dma(f, lev, comp, const_cast<double*>(host), true);
    double* stg = nullptr;
    CHK(stream_staging(h, (size_t)n, &stg));
    CU(cudaMemcpyAsync(stg, host, (size_t)n * 8, cudaMemcpyHostToDevice, t_stream));
    int err = PA_OK;
    const PaLayDev* ly = dev_layout(h, lev, f->ng, &err);
    if (!ly) return err;
    CU(launch_unpack_valid(D.boxes.p, ly, D.host_off.p, (int)h->H.lev[lev].local.size(), n, stg,
                           f->slab[lev] + (long long)comp * f->cs[lev], t_stream));
    return PA_OK;
}
int pa_field_download_level(const pa_field* f, int lev, int comp, double* host) {
    if (!f || lev < 0 || lev >= f->h->H.nlev || comp < 0 || comp >= f->ncomp || !host) return fail(PA_ERR_ARG, "pa_field_download_level: bad argument");
    pa_hier* h = f->h;
    LevelDev& D = *h->lev[lev];
    long long n = D.host_off_h.back();
    if (n == 0) return PA_OK;
    if (level_uses_dma(h, lev)) return level_dma(f, lev, comp, host, false);
    double* stg = nullptr;
    CHK(stream_staging(h, (size_t)n, &stg));
    int err = PA_OK;
    const PaLayDev* ly = dev_layout(h, lev, f->ng, &err);
    if (!ly) return err;
    CU(launch_pack_valid(D.boxes.p, ly, D.host_off.p, (int)h->H.lev[lev].local.size(), n,
                         f->slab[lev] + (long long)comp * f->cs[lev], stg, t_stream));
    CU(cudaMemcpyAsync(host, stg, (size_t)n * 8, cudaMemcpyDeviceToHost, t_stream));
    return PA_OK;
}
// ---- caller's device arrays (pa_array4) <-> valid cells of a level, one kernel launch per call ---------------------------
// Row items: a box is cut into runs of whole rows of about 4096 cells; the lanes sharing a row are the power of two (4..32)
// that the narrowest local box of the level fills, so 16-wide boxes keep all 32 lanes of a warp busy (two rows per warp).
static int device_io_items(pa_hier* h, int lev) {
    LevelDev& D = *h->lev[lev];
    if (!D.io_items_h.empty()) return PA_OK;
    const Level& V = h->H.lev[lev];
    int minx = 1 << 30;
    for (size_t lb = 0; lb < V.local.size(); ++lb) {
        const Box& B = V.boxes[V.local[lb]];
        minx = std::min(minx, B.len(0));
        const int rows = B.len(1) * B.len(2), per = std::max(1, 4096 / B.len(0));
        for (int r = 0; r < rows; r += per) D.io_items_h.push_back(PaRowItem{(int)lb, r, std::min(per, rows - r), 0});
    }
    D.io_lg_s = minx >= 32 ? 5 : minx >= 16 ? 4 : minx >= 8 ? 3 : 2;
    CU(D.io_items.upload(D.io_items_h, t_stream));      // the host vector lives as long as the hierarchy
    return PA_OK;
}

// Validates the arrays of one call and resolves them against the local boxes (records in local box order).
static int resolve_array4(const pa_field* f, int lev, int comp, int ncomp, const pa_array4* a, int na, bool is_dst, const char* who,
                          std::vector<PaA4Dev>& rec) {
    auto bad = [&](const std::string& m) { return fail(PA_ERR_ARG, std::string(who) + ": " + m); };
    if (!f || !f->h) return bad("null field");
    pa_hier* h = f->h;
    if (lev < 0 || lev >= h->H.nlev) return bad("level out of range");
    if (comp < 0 || ncomp < 1 || comp + ncomp > f->ncomp)
        return bad("field components [" + std::to_string(comp) + ", " + std::to_string(comp + ncomp) + ") out of [0, " + std::to_string(f->ncomp) + ")");
    const Level& V = h->H.lev[lev];
    if (na != (int)V.local.size())
        return bad("got " + std::to_string(na) + " arrays for the " + std::to_string(V.local.size()) + " boxes this rank owns on level " + std::to_string(lev));
    if (na > 0 && !a) return bad("null array list");
    int dev = 0;
    CU(cudaGetDevice(&dev));
    std::vector<std::pair<uintptr_t, uintptr_t>> ranges;
    rec.resize(na);
    for (int k = 0; k < na; ++k) {
        const pa_array4& A = a[k];
        const Box& B = V.boxes[V.local[k]];
        const std::string at = "array " + std::to_string(k) + " (global box " + std::to_string(V.local[k]) + "): ";
        if (!A.p) return bad(at + "null data pointer");
        for (int d = 0; d < 3; ++d)
            if (A.begin[d] > B.lo[d] || A.end[d] <= B.hi[d]) return bad(at + "begin / end do not contain the box");
        if (ncomp > A.ncomp) return bad(at + "ncomp " + std::to_string(ncomp) + " exceeds the array's " + std::to_string(A.ncomp) + " components");
        const long long lx = A.end[0] - A.begin[0], ly = A.end[1] - A.begin[1], lz = A.end[2] - A.begin[2];
        if (A.jstride < 0 || A.kstride < 0 || A.nstride < 0) return bad(at + "negative stride");
        if ((ly > 1 && A.jstride < lx) || (lz > 1 && A.kstride < (ly - 1) * A.jstride + lx) ||
            (A.ncomp > 1 && A.nstride < (lz - 1) * A.kstride + (ly - 1) * A.jstride + lx))
            return bad(at + "strides too small for the extents: rows, planes or components of the array overlap");
#if !defined(PA_HOST_EMULATION) || defined(PA_EMU_POINTER_ATTRIBUTES)
        cudaPointerAttributes pa;
        std::memset(&pa, 0, sizeof(pa));
        cudaError_t e = cudaPointerGetAttributes(&pa, A.p);
        if (e != cudaSuccess) { cudaGetLastError(); return bad(at + "cudaPointerGetAttributes failed: " + cudaGetErrorString(e)); }
        if (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged)
            return bad(at + "the pointer is host memory; host data goes through pa_field_upload_level / pa_field_download_level");
        if (pa.type == cudaMemoryTypeDevice && pa.device != dev)
            return bad(at + "the pointer is memory of device " + std::to_string(pa.device) + ", the calling thread's device is " + std::to_string(dev));
#else
        // a CPU test build whose runtime stand-in cannot tell device from host memory: refuse rather than guess
        return fail(PA_ERR_UNSUPPORTED, std::string(who) + ": this build cannot query pointer attributes");
#endif
        PaA4Dev& r = rec[k];
        r.p = A.p + (B.lo[0] - A.begin[0]) + (long long)(B.lo[1] - A.begin[1]) * A.jstride + (long long)(B.lo[2] - A.begin[2]) * A.kstride;
        r.js = A.jstride; r.ks = A.kstride; r.ns = A.nstride;
        if (is_dst) {
            const long long last = (B.len(0) - 1) + (long long)(B.len(1) - 1) * r.js + (long long)(B.len(2) - 1) * r.ks + (long long)(ncomp - 1) * r.ns;
            ranges.emplace_back((uintptr_t)r.p, (uintptr_t)(r.p + last + 1));
        }
    }
    if (is_dst) {
        std::vector<std::pair<uintptr_t, uintptr_t>> s = ranges;
        std::sort(s.begin(), s.end());
        for (size_t i = 1; i < s.size(); ++i)
            if (s[i].first < s[i - 1].second) return bad("destination arrays overlap: their written address ranges intersect");
    }
    return PA_OK;
}

static int device_copy(const pa_field* f, int lev, int comp, int ncomp, const pa_array4* a, int na, bool to_field, const char* who) {
    std::vector<PaA4Dev> rec;
    CHK(resolve_array4(f, lev, comp, ncomp, a, na, !to_field, who, rec));
    if (rec.empty()) return PA_OK;
    pa_hier* h = f->h;
    CHK(ensure_device(h));
    CHK(device_io_items(h, lev));
    auto& slot = h->a4[t_stream];
    if (!slot) {                       // sized for the level with the most local boxes: never reallocated afterwards
        slot = std::make_unique<DevBuf<PaA4Dev>>();
        size_t most = 1;
        for (const Level& V : h->H.lev) most = std::max(most, V.local.size());
        CU(slot->reserve(most));
    }
    // rec dies when this returns: a copy from pageable memory has been staged by the time cudaMemcpyAsync returns
    CU(cudaMemcpyAsync(slot->p, rec.data(), rec.size() * sizeof(PaA4Dev), cudaMemcpyHostToDevice, t_stream));
    int err = PA_OK;
    const PaLayDev* ly = dev_layout(h, lev, f->ng, &err);
    if (!ly) return err;
    LevelDev& D = *h->lev[lev];
    double* base = f->slab[lev] + (long long)comp * f->cs[lev];
    if (to_field) CU(launch_array4_to_field(D.io_items.p, (int)D.io_items_h.size(), D.boxes.p, ly, slot->p, ncomp, base, f->cs[lev], D.io_lg_s, t_stream));
    else CU(launch_field_to_array4(D.io_items.p, (int)D.io_items_h.size(), D.boxes.p, ly, slot->p, ncomp, base, f->cs[lev], D.io_lg_s, t_stream));
    return PA_OK;
}
int pa_field_upload_device(pa_field* f, int lev, int comp, int ncomp, const pa_array4* src, int nsrc) {
    return device_copy(f, lev, comp, ncomp, src, nsrc, true, "pa_field_upload_device");
}
int pa_field_download_device(const pa_field* f, int lev, int comp, int ncomp, const pa_array4* dst, int ndst) {
    return device_copy(f, lev, comp, ncomp, dst, ndst, false, "pa_field_download_device");
}

int pa_field_set_val(pa_field* f, int comp, int ncomp, double v) {
    CHK(check_field(f, comp, ncomp, "pa_field_set_val"));
    for (int l = 0; l < f->h->H.nlev; ++l)
        if (f->slab[l]) CU(launch_fill(f->slab[l] + (long long)comp * f->cs[l], f->cs[l] * ncomp, v, t_stream));
    return PA_OK;
}

int pa_field_hash(const pa_field* f, int comp, int ncomp, uint64_t* out) {
    CHK(check_field(f, comp, ncomp, "pa_field_hash"));
    if (!out) return fail(PA_ERR_ARG, "pa_field_hash: null result");
    pa_hier* h = f->h;
    CHK(ensure_device(h));
    unsigned long long* d = nullptr;
    CU(dev_alloc((void**)&d, sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(d, 0, sizeof(unsigned long long), t_stream);
    for (int l = 0; l < h->H.nlev && e == cudaSuccess; ++l) {
        const int nb = (int)h->H.lev[l].local.size();
        if (!nb) continue;
        int err = PA_OK;
        const PaLayDev* ly = dev_layout(h, l, f->ng, &err);
        if (!ly) { dev_free(d); return err; }
        e = launch_field_hash(h->lev[l]->boxes.p, ly, h->lev[l]->gid.p, nb, f->slab[l] + (long long)comp * f->cs[l], f->cs[l], comp, ncomp, l, d, t_stream);
    }
    unsigned long long v = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&v, d, sizeof(v), cudaMemcpyDeviceToHost, t_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(t_stream);
    dev_free(d);
    if (e != cudaSuccess) return cuda_fail(e, "pa_field_hash");
    *out = (uint64_t)v;
    return PA_OK;
}

// ---------------------------------------------------------------------------------------------- ghost cells
int pa_fill_boundary(pa_field* f, int comp, int ncomp, int cross) {
    CHK(check_field(f, comp, ncomp, "pa_fill_boundary"));
    pa_hier* h = f->h;
    Hier& H = h->H;
    CHK(ensure_device(h));
    if (f->ng < 1) return PA_OK;
    if (H.nranks > 1 && !cross) return fail(PA_ERR_UNSUPPORTED, "pa_fill_boundary(cross=0) is single-rank only");
    GridArgs ga;
    CHK(grid_args_inplace(f, comp, ga));
    const double* recv = nullptr;
    if (H.nranks > 1 && H.xplan.recv_prefix[H.nranks] + H.xplan.send_prefix[H.nranks] > 0) {
        if (f->recv_ncomp != ncomp || f->recv_comp0 != comp) return fail(PA_ERR_STATE, "exchange this component range first");
        recv = h->recv_slab.p;
    }
    if (f->peers_missing > 0) return fail(PA_ERR_STATE, "peer links: map every rank's slab of this field first (pa_field_map_peer)");
    for (int l = 0; l < H.nlev; ++l) {
        if (cross) {
            const HaloTable& T = H.halo_cross[l];
            CU(launch_halo(h->lev[l]->halo_cross.p, 0, (int)T.tags.size(), 0, T.ncells, ga.L[l].boxes, ga.L[l].lay_in, ga.L[l].out, f->cs[l], ncomp, recv,
                           ga.L[l].peers, comp, H.rank, GhostXform{0, 0.0, 1.0}, t_stream));
        } else {
            auto key = std::make_pair(l, f->ng);
            const HaloTable& T = H.halo_full(l, f->ng);
            auto it = h->halo_full.find(key);
            if (it == h->halo_full.end()) {
                auto buf = std::make_unique<DevBuf<PaHaloTag>>();
                CU(buf->upload(T.tags, t_stream));
                it = h->halo_full.emplace(key, std::move(buf)).first;
            }
            CU(launch_halo(it->second->p, 0, (int)T.tags.size(), 0, T.ncells, ga.L[l].boxes, ga.L[l].lay_in, ga.L[l].out, f->cs[l], ncomp, nullptr,
                           ga.L[l].peers, comp, H.rank, GhostXform{0, 0.0, 1.0}, t_stream));
        }
    }
    return PA_OK;
}

int pa_fill_ghosts(pa_field* f, int comp, int ncomp, int lev_lo, int lev_hi) {
    CHK(check_field(f, comp, ncomp, "pa_fill_ghosts"));
    if (lev_lo < 0) lev_lo = 0;
    if (lev_hi < 0 || lev_hi >= f->h->H.nlev) lev_hi = f->h->H.nlev - 1;
    if (lev_lo > lev_hi) return fail(PA_ERR_ARG, "pa_fill_ghosts: empty level range");
    return fill_ghosts_impl(f, comp, ncomp, lev_lo, lev_hi, true);
}

// ---------------------------------------------------------------------------------------------- exchange
int pa_exchange_counts(const pa_hier* h, int nghost, int ncomp, int64_t* send_counts, int64_t* recv_counts) {
    if (!h || !send_counts || !recv_counts || ncomp < 1) return fail(PA_ERR_ARG, "pa_exchange_counts: bad argument");
    (void)nghost;
    for (int p = 0; p < h->H.nranks; ++p) {
        send_counts[p] = (h->H.xplan.send_prefix[p + 1] - h->H.xplan.send_prefix[p]) * ncomp;
        recv_counts[p] = (h->H.xplan.recv_prefix[p + 1] - h->H.xplan.recv_prefix[p]) * ncomp;
    }
    return PA_OK;
}
int pa_exchange_buffers(pa_field* f, int ncomp, double** send_slab, double** recv_slab, int64_t* send_offsets, int64_t* recv_offsets) {
    if (!f || ncomp < 1) return fail(PA_ERR_ARG, "pa_exchange_buffers: bad argument");
    pa_hier* h = f->h;
    CHK(ensure_device(h));
    CHK(ensure_slabs(h, std::max(ncomp, h->slab_ncomp)));
    h->slab_ncomp = std::max(ncomp, h->slab_ncomp);
    if (send_slab) *send_slab = h->send_slab.p;
    if (recv_slab) *recv_slab = h->recv_slab.p;
    for (int p = 0; p <= h->H.nranks; ++p) {
        if (send_offsets) send_offsets[p] = h->H.xplan.send_prefix[p] * ncomp;
        if (recv_offsets) recv_offsets[p] = h->H.xplan.recv_prefix[p] * ncomp;
    }
    return PA_OK;
}
int pa_exchange_pack(pa_field* f, int comp, int ncomp) {
    CHK(check_field(f, comp, ncomp, "pa_exchange_pack"));
    pa_hier* h = f->h;
    Hier& H = h->H;
    CHK(ensure_device(h));
    f->recv_ncomp = 0;
    // the recv slab is shared by all fields of the hierarchy: the transport that follows this pack overwrites whatever another
    // field had received, so that field's mark must not survive (a later ghost fill on it would read this field's data)
    if (h->recv_owner && h->recv_owner != f) h->recv_owner->recv_ncomp = 0;
    h->recv_owner = nullptr;
    if (H.nranks <= 1) return PA_OK;
    CHK(ensure_slabs(h, std::max(ncomp, h->slab_ncomp)));
    h->slab_ncomp = std::max(ncomp, h->slab_ncomp);
    GridArgs ga;
    CHK(grid_args_inplace(f, comp, ga));
    long long ntags = (long long)H.xplan.pack.size();
    if (ntags) {
        const PaPackTag& last = H.xplan.pack.back();
        long long ncells = last.dense + (long long)last.n[0] * last.n[1] * last.n[2];
        CU(launch_exchange_pack(h->pack_tags.p, 0, ntags, 0, ncells, ga, ncomp, h->send_slab.p, t_stream));
    }
    return PA_OK;
}
int pa_exchange_mark_received(pa_field* f, int comp, int ncomp) {
    CHK(check_field(f, comp, ncomp, "pa_exchange_mark_received"));
    pa_hier* h = f->h;
    if (h->recv_owner && h->recv_owner != f) h->recv_owner->recv_ncomp = 0;
    h->recv_owner = f;
    f->recv_ncomp = ncomp;
    f->recv_comp0 = comp;
    return PA_OK;
}

// ---------------------------------------------------------------------------------------------- grad
int pa_grad(pa_field* in, int comp_in, int nvar, pa_field* out, int comp_out) {
    return pa_grad_phases(in, comp_in, nvar, out, comp_out, 3);
}

int pa_grad_phases(pa_field* in, int comp_in, int nvar, pa_field* out, int comp_out, int phases) {
    CHK(check_field(in, comp_in, nvar, "pa_grad(in)"));
    CHK(check_field(out, comp_out, 4 * nvar, "pa_grad(out)"));
    if (in->h != out->h) return fail(PA_ERR_ARG, "pa_grad: fields belong to different hierarchies");
    if (in->ng < 1) return fail(PA_ERR_ARG, "pa_grad: input field needs nghost >= 1");
    pa_hier* h = in->h;
    const int nlev = h->H.nlev;
    CHK(ensure_device(h));
    GridArgs ga;
    StencilExtra ex;
    std::memset(&ex, 0, sizeof(ex));
    if (phases == 3 && overlap_enabled(h)) {
        CHK(grid_args(in, comp_in, out, comp_out, ga));            // (also puts both layouts on the device before the fork)
        CHK(fill_ghosts_impl(in, comp_in, nvar, 0, 0, false));
        CHK(fork_side(h, [&]() { return fill_ghosts_impl(in, comp_in, nvar, 1, nlev - 1, false); }));
        CHK(run_stencil(h, MODE_GRAD, ga, ex, nvar, 0, 0, in->ng, in));
        CHK(join_side(h));
        return run_stencil(h, MODE_GRAD, ga, ex, nvar, 1, nlev - 1, in->ng, in);
    }
    if (phases & 1) CHK(fill_ghosts_impl(in, comp_in, nvar, 0, nlev - 1, false));
    if (!(phases & 2)) return PA_OK;
    CHK(grid_args(in, comp_in, out, comp_out, ga));
    return run_stencil(h, MODE_GRAD, ga, ex, nvar, 0, nlev - 1, in->ng, in);
}

// ---------------------------------------------------------------------------------------------- curvature
int pa_curvature_num_outputs(const pa_curv_opts* o) {
    if (!o) return 5;
    return 5 + (o->do_gauss ? 1 : 0) + (o->do_strain ? 1 : 0) + ((o->do_strain && o->get_strain_tensor) ? 9 : 0) + (o->do_velnormal ? 1 : 0);
}

static int tmp_field(pa_hier* h, pa_field** slot, int ncomp) {
    if (*slot && (*slot)->ncomp >= ncomp) return PA_OK;
    if (*slot) { pa_field_free(*slot); *slot = nullptr; }
    return pa_field_alloc(h, ncomp, 1, slot);
}

int pa_curvature(pa_field* state, int comp_S, int comp_vel, const pa_curv_opts* opts, pa_field* out, int comp_out) {
    if (state && state->h && state->h->H.nranks > 1)
        return fail(PA_ERR_UNSUPPORTED, "pa_curvature: on a multi-rank hierarchy the two passes are separated by a cross-rank step the caller "
                                        "owns; use pa_curvature_phases (1, exchange / barrier, 2)");
    return pa_curvature_phases(state, comp_S, comp_vel, opts, out, comp_out, 3);
}

// ---- the curvature tool, step by step -----------------------------------------------------------------------------
namespace {

// what every step needs: the two fields, the options and where each output lives in `out`
struct CurvCtx {
    pa_field* state; int comp_S, comp_vel;
    const pa_curv_opts* o;
    pa_field* out;
    pa_hier* h;
    int nlev;
    int cP, cK, cN, cKg, cSR, cROST, cVN;       // Progress, MeanCurvature, FlameNormalX.., optional outputs (-1: not enabled)
    double invdenom;
};

// The fused kernel (curv_fused.cu) serves the whole hierarchy or nothing: every local box must be eligible (build_curv_tiles).
// It is OPT-IN (PA_CURV_FUSED=1): measured on a B200 it moves a third less data than the separate NORMAL_S / DIV kernels
// (21.7 GB against 32.5 GB per step on the target hierarchy) but is bound by FP64 latency and per-SM store drain, not by HBM,
// and ends up slower (7.1 ms against 6.5 ms; DESIGN.md section 6 has the ablation).  The separate kernels are the default.
// PA_CURV_FUSED=3 selects the later fused kernel (curv_f3.cu: x strips, planes in shared memory) where every box is eligible
// for it (even width); the shell pass and the ghost fills are the same.  (PA_CURV_FUSED=2, curv_f2.cu, was its predecessor:
// measured 7.17 ms, superseded and removed.)  Returns 0 (separate kernels), 1 or 3.
int curv_fused_mode(const CurvCtx& c) {
    const char* e = getenv("PA_CURV_FUSED");
    const char* no_fuse = getenv("PA_CURV_UNFUSED");
    const char* es = getenv("PA_STENCIL");
    if (!(e && (e[0] == '1' || e[0] == '3')) || (no_fuse && no_fuse[0] == '1') || (es && !strcmp(es, "simple"))) return 0;
    if (!(c.state->ng == 1 && c.h->curv_ok && !overlap_enabled(c.h))) return 0;
    if (e[0] == '3') return (c.h->f3_ok && stencil_decide_normal_math(t_stream) == 0) ? 3 : 0;
    return 1;
}
bool curv_fused_path(const CurvCtx& c) { return curv_fused_mode(c) != 0; }

// PASS1: progress variable (curvature.cpp:310-321), its ghost cells, G = grad c, nrm, n = G / nrm (:426-502)
int curv_pass1(const CurvCtx& c) {
    pa_hier* h = c.h;
    Hier& H = h->H;
    const int nlev = c.nlev;
    StencilExtra ex;
    GridArgs ga;
    std::memset(&ex, 0, sizeof(ex));
    if (c.o->do_gauss) {                          // the Gaussian curvature needs the un-normalised gradient later
        CHK(tmp_field(h, &h->tmpG, 3));
        for (int l = 0; l < nlev; ++l) { ex.aux[l] = h->tmpG->slab[l]; ex.cs_aux[l] = h->tmpG->cs[l]; }
    }
    const char* no_fuse = getenv("PA_CURV_UNFUSED");
    if (curv_fused_path(c)) {
        // ONE kernel for Progress, the flame normal and K (curv_fused.cu): the ghost cells of S that must be materialised
        // (unlinked faces) are written in progress space first, as for MODE_NORMAL_S; K of the outermost cell layer of every
        // box follows in curv_div once the ghost cells of n exist.
        GhostXform xf{1, c.o->prog_min, c.invdenom};
        for (int l = 0; l < nlev; ++l) {
            ex.cout[l] = c.out->slab[l] ? c.out->slab[l] + (long long)c.cP * c.out->cs[l] : nullptr;
            ex.kout[l] = c.out->slab[l] ? c.out->slab[l] + (long long)c.cK * c.out->cs[l] : nullptr;
        }
        ex.pmin = c.o->prog_min; ex.inv = c.invdenom;
        ex.do_threshold = c.o->do_threshold ? 1 : 0;
        ex.threshold = c.o->threshold;
        CHK(grid_args(c.state, c.comp_S, c.out, c.cN, ga));
        if (c.state->peers_missing > 0)
            return fail(PA_ERR_STATE, "this hierarchy uses peer links (PA_HIER_PEER_LINKS): map every rank's slab of the state field first");
        CHK(fill_ghosts_impl(c.state, c.comp_S, 1, 0, nlev - 1, false, xf));
        if (curv_fused_mode(c) == 3) {
            TileTable& T = h->tiles_f3;
            const long long a = T.begin[0][0], b = T.begin[0][nlev];
            int lend[PA_MAX_LEVELS];
            for (int l = 0; l < nlev; ++l) lend[l] = (int)(T.begin[0][l + 1] - a);
            CU(launch_curv_f3(T.d.p + a, (int)(b - a), lend, nlev, ga, ex, t_stream));
            ++g_fused_launches;
            return PA_OK;
        }
        TileTable& T = h->tiles_curv;
        const long long a = T.begin[0][0], b = T.begin[0][nlev];
        CU(launch_curv_fused(T.d.p + a, (int)(b - a), T.max_plane_doubles, ga, ex, stencil_decide_normal_math(t_stream) != 0, t_stream));
        ++g_fused_launches;
        return PA_OK;
    }
    if (c.state->ng == 1 && use_tma(h, 1) && !(no_fuse && no_fuse[0] == '1')) {
        // Progress + normal fused.  The progress pass rides in the stencil's loader: valid cells stay S and are normalised as
        // they are read; the few ghost cells that must be materialised (unlinked faces) are written in progress space by the
        // ghost fill (coarse data = S on the next coarser level, normalised on load).  The kernel writes Progress and
        // n = G/nrm; Progress never makes a separate round trip through HBM.
        GhostXform xf{1, c.o->prog_min, c.invdenom};
        for (int l = 0; l < nlev; ++l) ex.cout[l] = c.out->slab[l] ? c.out->slab[l] + (long long)c.cP * c.out->cs[l] : nullptr;
        ex.pmin = c.o->prog_min; ex.inv = c.invdenom;
        CHK(grid_args(c.state, c.comp_S, c.out, c.cN, ga));
        if (overlap_enabled(h)) {
            CHK(fill_ghosts_impl(c.state, c.comp_S, 1, 0, 0, false, xf));
            CHK(fork_side(h, [&]() { return fill_ghosts_impl(c.state, c.comp_S, 1, 1, nlev - 1, false, xf); }));
            CHK(run_stencil(h, MODE_NORMAL_S, ga, ex, 1, 0, 0, c.state->ng, c.state));
            CHK(join_side(h));
            return run_stencil(h, MODE_NORMAL_S, ga, ex, 1, 1, nlev - 1, c.state->ng, c.state);
        }
        CHK(fill_ghosts_impl(c.state, c.comp_S, 1, 0, nlev - 1, false, xf));
        const char* nw = getenv("PA_NORMAL_W");
        if (nw && nw[0] == '1' && h->nw_ok && stencil_decide_normal_math(t_stream) == 0) {
            // S -> Progress, n through the barrier-free kernel of normal_w.cu (opt-in, same results)
            if (c.state->peers_missing > 0)
                return fail(PA_ERR_STATE, "this hierarchy uses peer links (PA_HIER_PEER_LINKS): map every rank's slab of the state field first");
            TileTable& T = h->tiles_nw;
            const long long a = T.begin[0][0], b = T.begin[0][nlev];
            CU(launch_normal_w(T.d.p + a, (int)(b - a), ga, ex, t_stream));
            ++g_fused_launches;
            return PA_OK;
        }
        const char* nf3 = getenv("PA_NORMAL_F3");
        if (nf3 && nf3[0] == '1' && h->n3_ok && stencil_decide_normal_math(t_stream) == 0) {
            // S -> Progress, n through the plane-staged kernel of curv_f3.cu without its K part (opt-in, same results)
            if (c.state->peers_missing > 0)
                return fail(PA_ERR_STATE, "this hierarchy uses peer links (PA_HIER_PEER_LINKS): map every rank's slab of the state field first");
            TileTable& T = h->tiles_n3;
            const long long a = T.begin[0][0], b = T.begin[0][nlev];
            int lend[PA_MAX_LEVELS];
            for (int l = 0; l < nlev; ++l) lend[l] = (int)(T.begin[0][l + 1] - a);
            CU(launch_normal_f3(T.d.p + a, (int)(b - a), lend, nlev, ga, ex, t_stream));
            ++g_fused_launches;
            return PA_OK;
        }
        return run_stencil(h, MODE_NORMAL_S, ga, ex, 1, 0, nlev - 1, c.state->ng, c.state);
    }
    if (H.nranks > 1)
        return fail(PA_ERR_UNSUPPORTED, "pa_curvature: the multi-rank path needs the fused progress pass (state with nghost == 1, "
                                        "TMA-eligible boxes); the unfused route would exchange an intermediate field");
    // unfused: c on valid cells of every level, ghost cells of c (coarse data = c on the next coarser level), then G -> nrm -> n
    for (int l = 0; l < nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* li = dev_layout(h, l, c.state->ng, &err);
        if (!li) return err;
        const PaLayDev* lo = dev_layout(h, l, c.out->ng, &err);
        if (!lo) return err;
        CU(launch_progress(h->lev[l]->boxes.p, li, lo, (int)H.lev[l].local.size(), c.state->slab[l] + (long long)c.comp_S * c.state->cs[l],
                           c.out->slab[l] + (long long)c.cP * c.out->cs[l], c.o->prog_min, c.invdenom, t_stream));
    }
    CHK(fill_ghosts_impl(c.out, c.cP, 1, 0, nlev - 1, false));
    CHK(grid_args(c.out, c.cP, c.out, c.cN, ga));
    return run_stencil(h, MODE_NORMAL, ga, ex, 1, 0, nlev - 1, c.out->ng, c.out);
}

// DIV: ghost cells of n, K = 0.5 div n (curvature.cpp:505-547) with the threshold clip of K (:549-567) on levels [l0, l1].
// After the fused PASS1 only the outermost cell layer of every box is left to do (k_div_shell).  The clip of n itself is a
// separate step (curv_clip): K of a level reads the UNCLIPPED n of that level (its own and, through neighbour links, other
// boxes' -- on a peer-linked hierarchy other ranks'), so n may only be clipped once every rank has finished DIV of the level.
// With the clip, level l needs the CLIPPED n of l-1 for its coarse-fine ghost cells (:514-518 reads flame_normal[lev-1]
// after :549-567 modified it), so the caller runs DIV(l), CLIP(l) level by level.
int curv_div(const CurvCtx& c, int l0, int l1) {
    pa_hier* h = c.h;
    pa_field* out = c.out;
    StencilExtra ex;
    GridArgs ga;
    std::memset(&ex, 0, sizeof(ex));
    ex.do_threshold = c.o->do_threshold ? 1 : 0;
    ex.threshold = c.o->threshold;
    for (int l = 0; l < c.nlev; ++l) ex.prog[l] = out->slab[l] + (long long)c.cP * out->cs[l];
    CHK(grid_args(out, c.cN, out, c.cK, ga));
    if (curv_fused_path(c)) {
        if (out->peers_missing > 0)
            return fail(PA_ERR_STATE, "this hierarchy uses peer links (PA_HIER_PEER_LINKS): map every rank's slab of the output field first");
        CHK(fill_ghosts_impl(out, c.cN, 3, l0, l1, false));
        const long long a = h->shell_begin[l0], b = h->shell_begin[l1 + 1];
        for (long long k = a; k < b; k += 65535) {
            const int n = (int)std::min<long long>(65535, b - k);
            CU(launch_div_shell(h->shell_level.p + k, h->shell_box.p + k, n, 24, ga, ex, t_stream));
            ++g_fused_launches;
        }
        return PA_OK;
    }
    if (overlap_enabled(h) && l0 == 0 && l1 > 0 && !c.o->do_threshold) {
        // n of every level is final: PASS1 is complete on the caller's stream, which the fork orders the side stream after
        CHK(fill_ghosts_impl(out, c.cN, 3, 0, 0, false));
        CHK(fork_side(h, [&]() { return fill_ghosts_impl(out, c.cN, 3, 1, l1, false); }));
        CHK(run_stencil(h, MODE_DIV, ga, ex, 1, 0, 0, out->ng, out));
        CHK(join_side(h));
        return run_stencil(h, MODE_DIV, ga, ex, 1, 1, l1, out->ng, out);
    }
    CHK(fill_ghosts_impl(out, c.cN, 3, l0, l1, false));
    return run_stencil(h, MODE_DIV, ga, ex, 1, l0, l1, out->ng, out);
}

// CLIP: n = 0 where the progress variable is outside [threshold, 1 - threshold] (curvature.cpp:549-567), levels [l0, l1]
int curv_clip(const CurvCtx& c, int l0, int l1) {
    pa_hier* h = c.h;
    Hier& H = h->H;
    pa_field* out = c.out;
    for (int l = l0; l <= l1; ++l) {
        int err = PA_OK;
        const PaLayDev* lo = dev_layout(h, l, out->ng, &err);
        if (!lo) { if (H.lev[l].local.empty()) continue; return err; }
        CU(launch_clip_normal(h->lev[l]->boxes.p, lo, lo, (int)H.lev[l].local.size(), out->slab[l] + (long long)c.cP * out->cs[l],
                              out->slab[l] + (long long)c.cN * out->cs[l], out->cs[l], c.o->threshold, t_stream));
    }
    return PA_OK;
}

// GAUSS: Hessian rows = grad3 of each un-normalised gradient component (ghosts by the same rules, coarse = G on l-1), then
// the pointwise n.adj(H).n / |grad c|^4 (curvature.cpp:575-677)
int curv_gauss(const CurvCtx& c) {
    pa_hier* h = c.h;
    Hier& H = h->H;
    if (!h->tmpG) return fail(PA_ERR_STATE, "pa_curvature_steps: PA_CURV_GAUSS before PA_CURV_PASS1");
    CHK(tmp_field(h, &h->tmpH, 9));
    CHK(fill_ghosts_impl(h->tmpG, 0, 3, 0, c.nlev - 1, false));
    StencilExtra e0;
    GridArgs ga;
    std::memset(&e0, 0, sizeof(e0));
    for (int d = 0; d < 3; ++d) {
        CHK(grid_args(h->tmpG, d, h->tmpH, 3 * d, ga));
        CHK(run_stencil(h, MODE_GRAD3, ga, e0, 1, 0, c.nlev - 1, h->tmpG->ng, h->tmpG));
    }
    for (int l = 0; l < c.nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* ly = dev_layout(h, l, 1, &err);
        if (!ly) return err;
        CU(launch_gauss(h->lev[l]->boxes.p, ly, ly, (int)H.lev[l].local.size(), h->tmpG->slab[l], h->tmpG->cs[l], h->tmpH->slab[l],
                        h->tmpH->cs[l], c.out->slab[l] + (long long)c.cP * c.out->cs[l], c.out->slab[l] + (long long)c.cKg * c.out->cs[l],
                        c.o->do_threshold ? 1 : 0, c.o->threshold, t_stream));
    }
    return PA_OK;
}

// STRAIN: velocity gradients with ghosts of u_i by the same rules (curvature.cpp:686-717), StrainRate and, on request, the
// nine ROST components (:719-759)
int curv_strain(const CurvCtx& c) {
    pa_hier* h = c.h;
    Hier& H = h->H;
    CHK(fill_ghosts_impl(c.state, c.comp_vel, 3, 0, c.nlev - 1, false));
    pa_field* dU = nullptr;
    int c0 = 0;
    if (c.cROST >= 0) { dU = c.out; c0 = c.cROST; }
    else { CHK(tmp_field(h, &h->tmpW, 9)); dU = h->tmpW; }
    StencilExtra e0;
    GridArgs ga;
    std::memset(&e0, 0, sizeof(e0));
    for (int d = 0; d < 3; ++d) {
        CHK(grid_args(c.state, c.comp_vel + d, dU, c0 + 3 * d, ga));
        CHK(run_stencil(h, MODE_GRAD3, ga, e0, 1, 0, c.nlev - 1, c.state->ng, c.state));
    }
    for (int l = 0; l < c.nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* ly = dev_layout(h, l, 1, &err);
        if (!ly) return err;
        CU(launch_strain(h->lev[l]->boxes.p, ly, (int)H.lev[l].local.size(), dU->slab[l] + (long long)c0 * dU->cs[l], dU->cs[l],
                         c.out->slab[l] + (long long)c.cSR * c.out->cs[l], t_stream));
    }
    return PA_OK;
}

// VELN: u . n with the (already clipped) normal (curvature.cpp:761-789), pointwise
int curv_veln(const CurvCtx& c) {
    pa_hier* h = c.h;
    Hier& H = h->H;
    for (int l = 0; l < c.nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* lu = dev_layout(h, l, c.state->ng, &err);
        if (!lu) return err;
        const PaLayDev* lo = dev_layout(h, l, 1, &err);
        if (!lo) return err;
        CU(launch_velnormal(h->lev[l]->boxes.p, lu, lo, lo, (int)H.lev[l].local.size(), c.state->slab[l] + (long long)c.comp_vel * c.state->cs[l],
                            c.state->cs[l], c.out->slab[l] + (long long)c.cN * c.out->cs[l], c.out->cs[l],
                            c.out->slab[l] + (long long)c.cP * c.out->cs[l], c.out->slab[l] + (long long)c.cVN * c.out->cs[l],
                            c.o->do_threshold ? 1 : 0, c.o->threshold, t_stream));
    }
    return PA_OK;
}

}  // namespace

// Single-rank callers run all steps in one call (pa_curvature); a multi-rank caller runs them one at a time with its
// cross-rank step (slab exchange and / or a barrier) in front of each -- the reference does the same through MPI inside
// FillBoundary / ParallelCopy (curvature.cpp:322, 487-502, 514-520, 686-717).  What each step needs exchanged:
//   PA_CURV_PASS1  S          PA_CURV_DIV  n (with threshold_prog: one level per call, in order)
//   PA_CURV_GAUSS  G (scratch field 0)      PA_CURV_STRAIN  the velocities      PA_CURV_VELN  nothing
int pa_curvature_steps(pa_field* state, int comp_S, int comp_vel, const pa_curv_opts* opts, pa_field* out, int comp_out, int steps,
                       int lev_lo, int lev_hi) {
    if (!opts) return fail(PA_ERR_ARG, "pa_curvature: null options");
    if (steps < 1 || steps > 63) return fail(PA_ERR_ARG, "pa_curvature_steps: steps must be a combination of PA_CURV_*");
    CHK(check_field(state, comp_S, 1, "pa_curvature(state)"));
    CHK(check_field(out, comp_out, pa_curvature_num_outputs(opts), "pa_curvature(out)"));
    if (state->h != out->h) return fail(PA_ERR_ARG, "pa_curvature: fields belong to different hierarchies");
    if (out->ng != 1) return fail(PA_ERR_ARG, "pa_curvature: the output field must have nghost == 1 (Progress and the flame normal are ghost-filled in place)");
    if (state->ng < 1) return fail(PA_ERR_ARG, "pa_curvature: state needs nghost >= 1");
    if (!(opts->prog_min < opts->prog_max)) return fail(PA_ERR_ARG, "progMin must be less than progMax");   // curvature.cpp:157-159
    if (opts->do_strain || opts->do_velnormal) CHK(check_field(state, comp_vel, 3, "pa_curvature(velocity)"));
    CurvCtx c;
    c.state = state; c.comp_S = comp_S; c.comp_vel = comp_vel; c.o = opts; c.out = out;
    c.h = state->h;
    CHK(ensure_device(c.h));
    c.nlev = c.h->H.nlev;
    if (lev_lo < 0) lev_lo = 0;
    if (lev_hi < 0 || lev_hi >= c.nlev) lev_hi = c.nlev - 1;
    if (lev_lo > lev_hi) return fail(PA_ERR_ARG, "pa_curvature_steps: empty level range");
    c.cP = comp_out; c.cK = comp_out + 1; c.cN = comp_out + 2;
    int next = comp_out + 5;
    c.cKg = opts->do_gauss ? next++ : -1;
    c.cSR = opts->do_strain ? next++ : -1;
    c.cROST = -1;
    if (opts->do_strain && opts->get_strain_tensor) { c.cROST = next; next += 9; }
    c.cVN = opts->do_velnormal ? next++ : -1;
    c.invdenom = 1.0 / (opts->prog_max - opts->prog_min);

    if (steps & PA_CURV_PASS1) CHK(curv_pass1(c));
    if ((steps & (PA_CURV_DIV | PA_CURV_CLIP)) && opts->do_threshold) {
        if (c.h->H.nranks > 1 && (lev_lo != lev_hi || (steps & (PA_CURV_DIV | PA_CURV_CLIP)) == (PA_CURV_DIV | PA_CURV_CLIP)))
            return fail(PA_ERR_ARG, "pa_curvature_steps: with threshold_prog a multi-rank caller runs PA_CURV_DIV and PA_CURV_CLIP one level "
                                    "per call, each in a call of its own (exchange the flame normal before DIV; every rank must have "
                                    "finished DIV of the level before any rank clips it)");
        // level by level: K of level l reads the unclipped n of l and the clipped n of l-1
        for (int l = lev_lo; l <= lev_hi; ++l) {
            if (steps & PA_CURV_DIV) CHK(curv_div(c, l, l));
            if (steps & PA_CURV_CLIP) CHK(curv_clip(c, l, l));
        }
    } else if (steps & PA_CURV_DIV) {
        CHK(curv_div(c, lev_lo, lev_hi));
    }
    if ((steps & PA_CURV_GAUSS) && opts->do_gauss) CHK(curv_gauss(c));
    if ((steps & PA_CURV_STRAIN) && opts->do_strain) CHK(curv_strain(c));
    if ((steps & PA_CURV_VELN) && opts->do_velnormal) CHK(curv_veln(c));
    return PA_OK;
}

int pa_curvature_phases(pa_field* state, int comp_S, int comp_vel, const pa_curv_opts* opts, pa_field* out, int comp_out, int phases) {
    if (!opts) return fail(PA_ERR_ARG, "pa_curvature: null options");
    if (phases < 1 || phases > 3) return fail(PA_ERR_ARG, "pa_curvature_phases: phases must be 1, 2 or 3");
    if (state && state->h && state->h->H.nranks > 1 && (opts->do_threshold || opts->do_gauss || opts->do_strain))
        return fail(PA_ERR_UNSUPPORTED, "pa_curvature_phases: threshold_prog / do_gaussCurv / do_strain need further cross-rank steps "
                                        "(per level, and of internal fields): use pa_curvature_steps");
    int steps = 0;
    if (phases & 1) steps |= PA_CURV_PASS1;
    if (phases & 2) steps |= PA_CURV_DIV | PA_CURV_CLIP | PA_CURV_GAUSS | PA_CURV_STRAIN | PA_CURV_VELN;
    return pa_curvature_steps(state, comp_S, comp_vel, opts, out, comp_out, steps, 0, -1);
}

// Internal field of the curvature tool a multi-rank caller has to exchange (and, with peer links, map): which = 0 the
// un-normalised gradient G of the progress variable (3 components, nghost 1; exists when do_gaussCurv is set, after
// PA_CURV_PASS1 ran once or after this call).  Owned by the hierarchy: do not free it.
int pa_curvature_scratch(pa_hier* h, int which, pa_field** f) {
    if (!h || !f || which != 0) return fail(PA_ERR_ARG, "pa_curvature_scratch: bad argument");
    CHK(ensure_device(h));
    CHK(tmp_field(h, &h->tmpG, 3));
    *f = h->tmpG;
    return PA_OK;
}

// ---- do_smooth: one backward-Euler diffusion step of the progress variable (curvature.cpp:328-406) --------------------------
}  // extern "C"
namespace {

// Order of the coarse-fine ghost polynomial of the smoothing operator.  AMReX's MLLinOp default maxorder is 3
// (AMReX_MLLinOp.H, LPInfo / maxorder); the gradient passes of the tools call setMaxOrder(4) (grad.cpp:179,
// curvature.cpp:426-441).  Whether curvature.cpp:328-406 calls setMaxOrder on its MLABecLaplacian is not verified here
// (DESIGN.md section 10, point 1): 3 holds unless it does.
constexpr int SMOOTH_MAXORDER = 3;
constexpr double SMOOTH_TOL_REL = 1e-10;
constexpr int SMOOTH_MAX_ITER = 1000;
// The multigrid preconditioner's V-cycle: red-black Gauss-Seidel sweeps before (NU1) and after (NU2) the coarse correction on
// every level, and a fixed number of sweeps on the coarsest coarsening of level 0 in place of a coarse solve.  Fixed counts and
// no tolerance: the V-cycle is the same linear map on every call, as right-preconditioned BiCGStab needs.
constexpr int SMOOTH_MG_NU1 = 2;
constexpr int SMOOTH_MG_NU2 = 2;
constexpr int SMOOTH_MG_BOTTOM_SWEEPS = 16;

// one level the V-cycle smooths: an AMR level of the hierarchy, or a coarsening of level 0 (level 0 of its own hierarchy)
struct SmLev {
    pa_hier* h;
    int l;
    const PaFaceRec* recs;              // face records of the ghost fill (nullptr: the hierarchy's own)
    const PaLayDev* lay;                // nghost-1 layout
    pa_field *e, *rhs, *res;            // correction, right-hand side, residual
};

struct SmCtx {
    pa_hier* h;
    SmoothDev* S;
    const SmoothTables* T;
    double beta;
    int nlev;
    std::vector<const PaLayDev*> lay;   // nghost-1 layout per level (every work field)
    bool mg = false;                    // preconditioner: the V-cycle (else Jacobi)
    std::vector<SmLev> amr;             // per AMR level (mg only; e is the V-cycle's output field)
    std::vector<SmLev> coarse;          // MG levels 1, 2, ... of level 0 (mg only)
};

// y = A x on every valid cell: covered cells of x <- fine averages, ghost fill, 7-point operator, reflux; y's covered cells <- 0
int sm_matvec(SmCtx& c, pa_field* x, pa_field* y) {
    pa_hier* h = c.h;
    Hier& H = h->H;
    const SmoothTables& T = *c.T;
    for (int l = c.nlev - 2; l >= 0; --l)
        CU(launch_sm_avgdown(c.S->avg.p + T.avg_begin[l], (int)(T.avg_begin[l + 1] - T.avg_begin[l]), T.avg_cells[l], h->lev[l]->boxes.p,
                             c.lay[l], h->lev[l + 1]->boxes.p, c.lay[l + 1], x->slab[l], x->slab[l + 1], false, t_stream));
    CHK(fill_ghosts_impl(x, 0, 1, 0, c.nlev - 1, true, GhostXform{0, 0.0, 1.0}, c.S->recs.p));
    for (int l = 0; l < c.nlev; ++l) {
        const LevelDev& D = *h->lev[l];
        CU(launch_sm_apply(D.boxes.p, c.lay[l], D.host_off.p, (int)H.lev[l].local.size(), D.host_off_h.back(), x->slab[l], y->slab[l],
                           c.beta, H.lev[l].dxinv, t_stream));
    }
    for (int l = 0; l + 1 < c.nlev; ++l)
        for (int g = 0; g < 6; ++g) {
            const long long a = T.reflux_begin[(size_t)l * 6 + g], b = T.reflux_begin[(size_t)l * 6 + g + 1];
            const int d = g / 2;
            CU(launch_sm_reflux(c.S->reflux.p + a, b - a, c.lay[l], c.lay[l + 1], x->slab[l], x->slab[l + 1], y->slab[l], c.beta,
                                H.lev[l].dxinv[d], H.lev[l + 1].dxinv[d], t_stream));
        }
    for (int l = 0; l + 1 < c.nlev; ++l)
        CU(launch_sm_avgdown(c.S->avg.p + T.avg_begin[l], (int)(T.avg_begin[l + 1] - T.avg_begin[l]), T.avg_cells[l], h->lev[l]->boxes.p,
                             c.lay[l], h->lev[l + 1]->boxes.p, c.lay[l + 1], y->slab[l], nullptr, true, t_stream));
    return PA_OK;
}

// out = a_l*x + b*y + cz*z on every level (whole slabs); a_l per level
int sm_lin(SmCtx& c, const std::vector<double>& a, pa_field* x, double b, pa_field* y, double cz, pa_field* z, pa_field* out) {
    for (int l = 0; l < c.nlev; ++l)
        CU(launch_sm_lin3(out->cs[l], a[l], x->slab[l], b, y ? y->slab[l] : nullptr, cz, z ? z->slab[l] : nullptr, out->slab[l], t_stream));
    return PA_OK;
}

// mode 0: sum over valid cells of x*y; mode 1: max |x| (NaN if any cell is NaN).  Fixed reduction order; synchronises.
int sm_reduce(SmCtx& c, pa_field* x, pa_field* y, int mode, double* out) {
    int off = 0;
    for (int l = 0; l < c.nlev; ++l) {
        const LevelDev& D = *c.h->lev[l];
        int nb = 0;
        CU(launch_sm_reduce(D.boxes.p, c.lay[l], D.host_off.p, (int)c.h->H.lev[l].local.size(), D.host_off_h.back(), x->slab[l],
                            y ? y->slab[l] : nullptr, mode, c.S->partial.p + off, &nb, t_stream));
        off += nb;
    }
    CU(launch_sm_final(c.S->partial.p, off, mode, c.S->scal.p, t_stream));
    CU(cudaMemcpyAsync(out, c.S->scal.p, sizeof(double), cudaMemcpyDeviceToHost, t_stream));
    CU(cudaStreamSynchronize(t_stream));
    return PA_OK;
}

// ---- the multigrid preconditioner -----------------------------------------------------------------------------------------
int sm_fill(const SmLev& v) { return fill_ghosts_impl(v.e, 0, 1, v.l, v.l, true, GhostXform{0, 0.0, 1.0}, v.recs); }

// n red-black Gauss-Seidel sweeps of A_l e = rhs on one level; the ghost cells are refilled before each colour
int sm_gsrb(const SmLev& v, double beta, int n) {
    const LevelDev& D = *v.h->lev[v.l];
    const Level& V = v.h->H.lev[v.l];
    const double* q = V.dxinv;
    const double diag = 1.0 + 2.0 * beta * (q[0] * q[0] + q[1] * q[1] + q[2] * q[2]);
    for (int s = 0; s < n; ++s)
        for (int colour = 0; colour < 2; ++colour) {
            CHK(sm_fill(v));
            CU(launch_sm_gsrb(D.boxes.p, v.lay, D.host_off.p, (int)V.local.size(), D.host_off_h.back(), v.rhs->slab[v.l], v.e->slab[v.l],
                              beta, q, diag, colour, t_stream));
        }
    return PA_OK;
}

// res = rhs - A_l e on one level (ghost cells refilled first)
int sm_resid(const SmLev& v, double beta) {
    const LevelDev& D = *v.h->lev[v.l];
    const Level& V = v.h->H.lev[v.l];
    CHK(sm_fill(v));
    CU(launch_sm_resid(D.boxes.p, v.lay, D.host_off.p, (int)V.local.size(), D.host_off_h.back(), v.rhs->slab[v.l], v.e->slab[v.l],
                       v.res->slab[v.l], beta, V.dxinv, t_stream));
    return PA_OK;
}

int sm_zero(pa_field* f, int l) {
    if (f->cs[l] > 0) CU(cudaMemsetAsync(f->slab[l], 0, (size_t)f->cs[l] * sizeof(double), t_stream));
    return PA_OK;
}

// z = B r, one V-cycle from a zero initial guess (DESIGN.md section 10):
//  1. AMR levels L .. 1: NU1 sweeps, the residual, restricted into level l-1 -- the 8-cell average on covered cells, and on the
//     uncovered coarse cells of coarse-fine faces minus the fine-flux term of the composite operator (the reflux of z_l
//     against a zero z_{l-1}, i.e. with beta negated);
//  2. level 0: a geometric V-cycle over its coarsenings (8-cell average down, piecewise-constant up, NU1 / NU2 sweeps, the
//     coarsest level SMOOTH_MG_BOTTOM_SWEEPS sweeps);
//  3. AMR levels 1 .. L: z_l += the piecewise-constant prolongation of z_{l-1}, NU2 sweeps with ghost cells from z_{l-1};
//  4. covered cells of z <- 0 (the Krylov vectors are zero there).
int sm_vcycle(SmCtx& c, pa_field* r, pa_field* z) {
    pa_hier* h = c.h;
    const Hier& H = h->H;
    const SmoothTables& T = *c.T;
    SmoothDev& S = *c.S;
    const int L = c.nlev - 1;
    for (int l = 0; l <= L; ++l) {
        c.amr[l].e = z;
        CHK(sm_zero(z, l));
        CU(launch_sm_lin3(r->cs[l], 1.0, r->slab[l], 0.0, nullptr, 0.0, nullptr, S.mg_rhs->slab[l], t_stream));
    }
    for (int l = L; l >= 1; --l) {
        const SmLev& v = c.amr[l];
        CHK(sm_gsrb(v, c.beta, SMOOTH_MG_NU1));
        CHK(sm_resid(v, c.beta));
        CU(launch_sm_avgdown(S.avg.p + T.avg_begin[l - 1], (int)(T.avg_begin[l] - T.avg_begin[l - 1]), T.avg_cells[l - 1],
                             h->lev[l - 1]->boxes.p, c.lay[l - 1], h->lev[l]->boxes.p, c.lay[l], S.mg_rhs->slab[l - 1], S.mg_res->slab[l],
                             false, t_stream));
        for (int g = 0; g < 6; ++g) {
            const long long a = T.reflux_begin[(size_t)(l - 1) * 6 + g], b = T.reflux_begin[(size_t)(l - 1) * 6 + g + 1];
            const int d = g / 2;
            CU(launch_sm_reflux(S.reflux.p + a, b - a, c.lay[l - 1], c.lay[l], z->slab[l - 1], z->slab[l], S.mg_rhs->slab[l - 1], -c.beta,
                                H.lev[l - 1].dxinv[d], H.lev[l].dxinv[d], t_stream));
        }
    }
    const int K = 1 + (int)c.coarse.size();
    auto mg = [&](int k) -> const SmLev& { return k == 0 ? c.amr[0] : c.coarse[k - 1]; };
    for (int k = 0; k + 1 < K; ++k) {
        const SmLev &f = mg(k), &q = mg(k + 1);
        CHK(sm_gsrb(f, c.beta, SMOOTH_MG_NU1));
        CHK(sm_resid(f, c.beta));
        CHK(sm_zero(q.e, 0));
        CU(launch_sm_avgdown(S.mg_avg.p + T.mg_avg_begin[k], (int)(T.mg_avg_begin[k + 1] - T.mg_avg_begin[k]), T.mg_avg_cells[k],
                             q.h->lev[0]->boxes.p, q.lay, f.h->lev[f.l]->boxes.p, f.lay, q.rhs->slab[0], f.res->slab[f.l], false, t_stream));
    }
    CHK(sm_gsrb(mg(K - 1), c.beta, SMOOTH_MG_BOTTOM_SWEEPS));
    for (int k = K - 2; k >= 0; --k) {
        const SmLev &f = mg(k), &q = mg(k + 1);
        CU(launch_sm_prolong(S.mg_avg.p + T.mg_avg_begin[k], (int)(T.mg_avg_begin[k + 1] - T.mg_avg_begin[k]), T.mg_avg_cells[k],
                             q.h->lev[0]->boxes.p, q.lay, f.h->lev[f.l]->boxes.p, f.lay, q.e->slab[0], f.e->slab[f.l], t_stream));
        CHK(sm_gsrb(f, c.beta, SMOOTH_MG_NU2));
    }
    for (int l = 1; l <= L; ++l) {
        CU(launch_sm_prolong(S.avg.p + T.avg_begin[l - 1], (int)(T.avg_begin[l] - T.avg_begin[l - 1]), T.avg_cells[l - 1],
                             h->lev[l - 1]->boxes.p, c.lay[l - 1], h->lev[l]->boxes.p, c.lay[l], z->slab[l - 1], z->slab[l], t_stream));
        CHK(sm_gsrb(c.amr[l], c.beta, SMOOTH_MG_NU2));
    }
    for (int l = 0; l < L; ++l)
        CU(launch_sm_avgdown(S.avg.p + T.avg_begin[l], (int)(T.avg_begin[l + 1] - T.avg_begin[l]), T.avg_cells[l], h->lev[l]->boxes.p,
                             c.lay[l], h->lev[l + 1]->boxes.p, c.lay[l + 1], z->slab[l], nullptr, true, t_stream));
    return PA_OK;
}

int ensure_smooth(pa_hier* h, const SmoothTables& T) {
    if (h->sm) return PA_OK;
    auto S = std::make_unique<SmoothDev>();
    CU(S->recs.upload(T.recs, t_stream));
    CU(S->avg.upload(T.avg, t_stream));
    CU(S->reflux.upload(T.reflux, t_stream));
    CU(S->partial.reserve((size_t)std::max(1, h->H.nlev) * smooth_max_partials()));
    CU(S->scal.reserve(1));
    CU(cudaStreamSynchronize(t_stream));
    for (auto& f : S->w) {
        int rc = pa_field_alloc(h, 1, 1, &f);
        if (rc != PA_OK) { for (pa_field* g : S->w) if (g) pa_field_free(g); return rc; }
    }
    h->sm = std::move(S);
    return PA_OK;
}

// the multigrid preconditioner's work fields and level-0 coarsenings: one single-level, one-rank hierarchy per coarsening
// (boxes and domain of T.mg_boxes / T.mg_dom, dx * 2^k, the hierarchy's periodicity and wall kinds), which brings its layouts,
// halo and wall tables and ghost fill
int ensure_smooth_mg(pa_hier* h, const SmoothTables& T) {
    SmoothDev& S = *h->sm;
    if (S.mg_ready) return PA_OK;
    free_smooth_mg(S);                  // what an earlier, failed attempt left
    const Hier& H = h->H;
    CHK(pa_field_alloc(h, 1, 1, &S.mg_rhs));
    CHK(pa_field_alloc(h, 1, 1, &S.mg_res));
    for (size_t k = 1; k < T.mg_boxes.size(); ++k) {
        const std::vector<Box>& B = T.mg_boxes[k];
        std::vector<int> bx;
        for (const Box& b : B) bx.insert(bx.end(), {b.lo[0], b.lo[1], b.lo[2], b.hi[0], b.hi[1], b.hi[2]});
        pa_level_desc L{};
        for (int d = 0; d < 3; ++d) {
            L.domain_lo[d] = T.mg_dom[k].lo[d];
            L.domain_hi[d] = T.mg_dom[k].hi[d];
            L.dx[d] = H.lev[0].dx[d] * (double)(1 << k);
        }
        L.nboxes = (int)B.size();
        L.boxes = bx.data();
        L.owner = nullptr;
        pa_hier* m = nullptr;
        CHK(pa_hier_create2(&m, 1, &L, H.is_per, H.bc_kind, 0, 1, 0u));
        S.mg_h.push_back(m);
        S.mg_f.push_back({nullptr, nullptr, nullptr});
        for (pa_field*& f : S.mg_f.back()) CHK(pa_field_alloc(m, 1, 1, &f));
    }
    CU(S.mg_avg.upload(T.mg_avg, t_stream));
    CU(cudaStreamSynchronize(t_stream));
    S.mg_ready = true;
    return PA_OK;
}

// What pa_smooth and pa_debug_smooth_vcycle share: argument checks, tables, work fields (and, with mg, the multigrid
// preconditioner's), and c = (S - progMin) * invdenom -- pa_curvature's Progress arithmetic (curvature.cpp:310-321) -- into
// out[comp_c] and, for t > 0, into the right-hand side w[1]; for t = 0 into out[comp_phi] as well.
int smooth_prepare(pa_field* state, int comp_S, double prog_min, double prog_max, const pa_smooth_opts* o, pa_field* out, int comp_c,
                   int comp_phi, SmCtx& c) {
    if (!o) return fail(PA_ERR_ARG, "pa_smooth: null options");
    CHK(check_field(state, comp_S, 1, "pa_smooth(state)"));
    CHK(check_field(out, comp_c, 1, "pa_smooth(out, comp_c)"));
    CHK(check_field(out, comp_phi, 1, "pa_smooth(out, comp_phi)"));
    if (state->h != out->h) return fail(PA_ERR_ARG, "pa_smooth: fields belong to different hierarchies");
    if (comp_c == comp_phi) return fail(PA_ERR_ARG, "pa_smooth: comp_c and comp_phi must differ");
    if (out == state && (comp_c == comp_S || comp_phi == comp_S)) return fail(PA_ERR_ARG, "pa_smooth: the outputs would overwrite S");
    if (!(prog_min < prog_max)) return fail(PA_ERR_ARG, "progMin must be less than progMax");   // curvature.cpp:157-159
    const double t = o->smoothing_time;
    if (!(t >= 0.0) || !std::isfinite(t)) return fail(PA_ERR_ARG, "pa_smooth: smoothing_time must be finite and >= 0");
    if (!(o->tol_rel >= 0.0) || o->max_iter < 0) return fail(PA_ERR_ARG, "pa_smooth: tol_rel and max_iter must be >= 0 (0 = default)");
    if (o->precond != PA_SMOOTH_PRECOND_JACOBI && o->precond != PA_SMOOTH_PRECOND_MG)
        return fail(PA_ERR_ARG, "pa_smooth: unknown precond " + std::to_string(o->precond) + " (PA_SMOOTH_PRECOND_JACOBI = 0, PA_SMOOTH_PRECOND_MG = 1)");
    pa_hier* h = state->h;
    Hier& H = h->H;
    if (H.nranks > 1) return fail(PA_ERR_UNSUPPORTED, "pa_smooth supports one rank only (do_smooth is not available on several GPUs)");
    if (H.filter_only) return fail(PA_ERR_UNSUPPORTED, "pa_smooth needs a hierarchy created without PA_HIER_FILTER_ONLY");
    for (int l = 1; l < H.nlev; ++l)
        if (H.lev[l].ratio != 2)
            return fail(PA_ERR_UNSUPPORTED, "pa_smooth supports refinement ratio 2 only (curvature.cpp:445,518,842 hard-code it); level " +
                                                std::to_string(l) + " has ratio " + std::to_string(H.lev[l].ratio));
    CHK(ensure_device(h));
    const SmoothTables& T = H.smooth_tables(SMOOTH_MAXORDER);
    if (!T.err.empty()) return fail(PA_ERR_ARG, T.err);
    CHK(ensure_smooth(h, T));
    c.h = h; c.S = h->sm.get(); c.T = &T; c.beta = t; c.nlev = H.nlev;
    for (int l = 0; l < H.nlev; ++l) {
        int err = PA_OK;
        const PaLayDev* ly = dev_layout(h, l, 1, &err);
        if (!ly && !H.lev[l].local.empty()) return err;
        c.lay.push_back(ly);
    }
    c.mg = o->precond == PA_SMOOTH_PRECOND_MG;
    if (c.mg && t > 0.0) {
        CHK(ensure_smooth_mg(h, T));
        SmoothDev& S = *c.S;
        for (int l = 0; l < H.nlev; ++l) c.amr.push_back(SmLev{h, l, S.recs.p, c.lay[l], nullptr, S.mg_rhs, S.mg_res});
        for (size_t k = 0; k < S.mg_h.size(); ++k) {
            int err = PA_OK;
            const PaLayDev* ly = dev_layout(S.mg_h[k], 0, 1, &err);
            if (!ly) return err;
            c.coarse.push_back(SmLev{S.mg_h[k], 0, nullptr, ly, S.mg_f[k][0], S.mg_f[k][1], S.mg_f[k][2]});
        }
    }
    pa_field* b = c.S->w[1];
    const double invdenom = 1.0 / (prog_max - prog_min);
    for (int l = 0; l < H.nlev; ++l) {
        const LevelDev& D = *h->lev[l];
        const int nb = (int)H.lev[l].local.size();
        int err = PA_OK;
        const PaLayDev* ls = dev_layout(h, l, state->ng, &err);
        const PaLayDev* lo = dev_layout(h, l, out->ng, &err);
        if (nb && (!ls || !lo)) return err;
        const double* S = state->slab[l] + (long long)comp_S * state->cs[l];
        CU(launch_progress(D.boxes.p, ls, lo, nb, S, out->slab[l] + (long long)comp_c * out->cs[l], prog_min, invdenom, t_stream));
        if (t == 0.0)      // phi - 0 * Laplacian(phi) = c: phi is c, bit for bit
            CU(launch_progress(D.boxes.p, ls, lo, nb, S, out->slab[l] + (long long)comp_phi * out->cs[l], prog_min, invdenom, t_stream));
        else
            CU(launch_progress(D.boxes.p, ls, c.lay[l], nb, S, b->slab[l], prog_min, invdenom, t_stream));
    }
    return PA_OK;
}

// x = c (initial guess), then b's covered cells <- 0 (the right-hand side lives on the uncovered cells); *bmax = max|b|
int smooth_start(SmCtx& c, pa_field* x, pa_field* b, double* bmax) {
    const SmoothTables& T = *c.T;
    const std::vector<double> one(c.nlev, 1.0);
    CHK(sm_lin(c, one, b, 0.0, nullptr, 0.0, nullptr, x));
    for (int l = 0; l + 1 < c.nlev; ++l)
        CU(launch_sm_avgdown(c.S->avg.p + T.avg_begin[l], (int)(T.avg_begin[l + 1] - T.avg_begin[l]), T.avg_cells[l], c.h->lev[l]->boxes.p,
                             c.lay[l], c.h->lev[l + 1]->boxes.p, c.lay[l + 1], b->slab[l], nullptr, true, t_stream));
    CHK(sm_reduce(c, b, nullptr, 1, bmax));
    if (!std::isfinite(*bmax)) return fail(PA_ERR_ARG, "pa_smooth: the progress variable has non-finite values");
    return PA_OK;
}

// covered cells of phi <- fine averages, then phi -> out[comp_phi]
int smooth_finish(SmCtx& c, pa_field* x, pa_field* out, int comp_phi) {
    pa_hier* h = c.h;
    const Hier& H = h->H;
    const SmoothTables& T = *c.T;
    for (int l = H.nlev - 2; l >= 0; --l)
        CU(launch_sm_avgdown(c.S->avg.p + T.avg_begin[l], (int)(T.avg_begin[l + 1] - T.avg_begin[l]), T.avg_cells[l], h->lev[l]->boxes.p,
                             c.lay[l], h->lev[l + 1]->boxes.p, c.lay[l + 1], x->slab[l], x->slab[l + 1], false, t_stream));
    for (int l = 0; l < H.nlev; ++l) {
        const LevelDev& D = *h->lev[l];
        int err = PA_OK;
        const PaLayDev* lo = dev_layout(h, l, out->ng, &err);
        CU(launch_sm_copy(D.boxes.p, c.lay[l], lo, D.host_off.p, (int)H.lev[l].local.size(), D.host_off_h.back(), x->slab[l],
                          out->slab[l] + (long long)comp_phi * out->cs[l], t_stream));
    }
    return PA_OK;
}

}  // namespace
extern "C" {

int pa_smooth(pa_field* state, int comp_S, double prog_min, double prog_max, const pa_smooth_opts* o, pa_field* out, int comp_c,
              int comp_phi, int* iters, double* resid) {
    if (iters) *iters = 0;
    if (resid) *resid = 0.0;
    SmCtx c;
    CHK(smooth_prepare(state, comp_S, prog_min, prog_max, o, out, comp_c, comp_phi, c));
    const double t = c.beta;
    if (t == 0.0) return PA_OK;
    const double tol_rel = o->tol_rel > 0.0 ? o->tol_rel : SMOOTH_TOL_REL;
    const int max_iter = o->max_iter > 0 ? o->max_iter : SMOOTH_MAX_ITER;
    const int nlev = c.nlev;
    const Hier& H = c.h->H;
    pa_field **w = c.S->w, *x = w[0], *b = w[1], *r = w[2], *r0 = w[3], *p = w[4], *v = w[5], *tt = w[6], *z = w[7];
    const std::vector<double> one(nlev, 1.0), zero(nlev, 0.0);
    std::vector<double> jac(nlev);           // Jacobi preconditioner: the inverse diagonal of each level's operator
    for (int l = 0; l < nlev; ++l) {
        const double* q = H.lev[l].dxinv;
        jac[l] = 1.0 / (1.0 + 2.0 * t * (q[0] * q[0] + q[1] * q[1] + q[2] * q[2]));
    }
    // z = M^-1 y: the Jacobi scaling or one V-cycle
    auto precondition = [&](pa_field* y) -> int { return c.mg ? sm_vcycle(c, y, z) : sm_lin(c, jac, y, 0.0, nullptr, 0.0, nullptr, z); };
    double bmax = 0.0;
    CHK(smooth_start(c, x, b, &bmax));
    const double tol = tol_rel * bmax;
    // true residual r = b - A x
    auto true_residual = [&](double* rn) -> int {
        CHK(sm_matvec(c, x, tt));
        CHK(sm_lin(c, one, b, -1.0, tt, 0.0, nullptr, r));
        return sm_reduce(c, r, nullptr, 1, rn);
    };
    double rnorm = 0.0;
    CHK(true_residual(&rnorm));
    // Right-preconditioned BiCGStab on the composite operator, restarted from the true residual whenever the recurrence
    // residual meets the tolerance but the true one does not, or on a breakdown.
    int it = 0;
    bool restart = true;
    double rho_old = 1.0, alpha = 1.0, omega = 1.0;
    while (!(rnorm <= tol)) {
        if (it >= max_iter || !std::isfinite(rnorm)) {
            if (iters) *iters = it;
            if (resid) *resid = bmax > 0.0 ? rnorm / bmax : rnorm;
            char msg[256];
            std::snprintf(msg, sizeof msg, "pa_smooth: not converged after %d iterations: max|c - A phi| / max|c| = %.3e (tol_rel %.3e)", it,
                          bmax > 0.0 ? rnorm / bmax : rnorm, tol_rel);
            return fail(PA_ERR_NOCONV, msg);
        }
        if (restart) {
            CHK(sm_lin(c, one, r, 0.0, nullptr, 0.0, nullptr, r0));
            CHK(sm_lin(c, zero, r, 0.0, nullptr, 0.0, nullptr, p));
            CHK(sm_lin(c, zero, r, 0.0, nullptr, 0.0, nullptr, v));
            rho_old = alpha = omega = 1.0;
            restart = false;
        }
        ++it;
        double rho = 0.0;
        CHK(sm_reduce(c, r0, r, 0, &rho));
        if (rho == 0.0 || !std::isfinite(rho)) { restart = true; CHK(true_residual(&rnorm)); continue; }
        const double bk = (rho / rho_old) * (alpha / omega);
        CHK(sm_lin(c, one, r, bk, p, -bk * omega, v, p));                   // p = r + bk (p - omega v)
        CHK(precondition(p));                                                // z = M^-1 p
        CHK(sm_matvec(c, z, v));                                             // v = A z
        double den = 0.0;
        CHK(sm_reduce(c, r0, v, 0, &den));
        if (den == 0.0 || !std::isfinite(den)) { restart = true; CHK(true_residual(&rnorm)); continue; }
        alpha = rho / den;
        CHK(sm_lin(c, one, r, -alpha, v, 0.0, nullptr, r));                  // s = r - alpha v (in r)
        CHK(sm_lin(c, one, x, alpha, z, 0.0, nullptr, x));                   // x += alpha z
        double snorm = 0.0;
        CHK(sm_reduce(c, r, nullptr, 1, &snorm));
        rho_old = rho;
        if (!(snorm <= tol)) {
            CHK(precondition(r));                                            // z = M^-1 s
            CHK(sm_matvec(c, z, tt));                                        // t = A z
            double ts = 0.0, t2 = 0.0;
            CHK(sm_reduce(c, tt, r, 0, &ts));
            CHK(sm_reduce(c, tt, tt, 0, &t2));
            if (t2 == 0.0 || !std::isfinite(t2) || ts == 0.0) { restart = true; CHK(true_residual(&rnorm)); continue; }
            omega = ts / t2;
            CHK(sm_lin(c, one, x, omega, z, 0.0, nullptr, x));               // x += omega z
            CHK(sm_lin(c, one, r, -omega, tt, 0.0, nullptr, r));             // r = s - omega t
            CHK(sm_reduce(c, r, nullptr, 1, &snorm));
        }
        rnorm = snorm;
        if (rnorm <= tol) {                                                  // converged by the recurrence: confirm on the true residual
            CHK(true_residual(&rnorm));
            if (!(rnorm <= tol)) restart = true;
        }
    }
    CHK(smooth_finish(c, x, out, comp_phi));
    if (iters) *iters = it;
    if (resid) *resid = bmax > 0.0 ? rnorm / bmax : 0.0;
    return PA_OK;
}

int pa_debug_smooth_vcycle(pa_field* state, int comp_S, double prog_min, double prog_max, const pa_smooth_opts* o, pa_field* out,
                           int comp_c, int comp_phi, int ncycles, double* resid, int* nmg) {
    if (nmg) *nmg = 0;
    if (!o || !(o->smoothing_time > 0.0)) return fail(PA_ERR_ARG, "pa_debug_smooth_vcycle: needs options with smoothing_time > 0");
    if (ncycles < 0 || !resid) return fail(PA_ERR_ARG, "pa_debug_smooth_vcycle: ncycles must be >= 0 and resid non-null");
    pa_smooth_opts om = *o;
    om.precond = PA_SMOOTH_PRECOND_MG;
    SmCtx c;
    CHK(smooth_prepare(state, comp_S, prog_min, prog_max, &om, out, comp_c, comp_phi, c));
    if (nmg) *nmg = (int)c.T->mg_boxes.size();
    pa_field **w = c.S->w, *x = w[0], *b = w[1], *r = w[2], *tt = w[6], *z = w[7];
    const std::vector<double> one(c.nlev, 1.0);
    double bmax = 0.0;
    CHK(smooth_start(c, x, b, &bmax));
    for (int n = 0; n <= ncycles; ++n) {
        if (n > 0) {
            CHK(sm_vcycle(c, r, z));
            CHK(sm_lin(c, one, x, 1.0, z, 0.0, nullptr, x));               // phi += B r
        }
        CHK(sm_matvec(c, x, tt));
        CHK(sm_lin(c, one, b, -1.0, tt, 0.0, nullptr, r));                 // r = c - A phi
        double rn = 0.0;
        CHK(sm_reduce(c, r, nullptr, 1, &rn));
        resid[n] = bmax > 0.0 ? rn / bmax : rn;
    }
    return smooth_finish(c, x, out, comp_phi);
}

// ---------------------------------------------------------------------------------------------- debug
int pa_debug_fb_source_map(pa_hier* h, int lev, int nghost, int cross, int64_t* out, int64_t out_len) {
    if (!h || lev < 0 || lev >= h->H.nlev || !out) return fail(PA_ERR_ARG, "pa_debug_fb_source_map: bad argument");
    Hier& H = h->H;
    const Level& V = H.lev[lev];
    const HaloTable* T;
    HaloTable tmp;
    if (cross && nghost == 1) T = &H.halo_cross[lev];
    else if (!cross) { if (H.nranks > 1) return fail(PA_ERR_UNSUPPORTED, "single-rank only"); T = &H.halo_full(lev, nghost); }
    else return fail(PA_ERR_ARG, "cross tables exist for nghost == 1 only");
    std::vector<long long> off(V.local.size() + 1, 0);
    for (size_t lb = 0; lb < V.local.size(); ++lb) off[lb + 1] = off[lb] + V.boxes[V.local[lb]].grown(nghost).npts();
    if (out_len < off.back()) return fail(PA_ERR_ARG, "output buffer too small");
    std::fill(out, out + off.back(), (int64_t)-1);
    for (const PaHaloTag& t : T->tags) {
        const Box g = V.boxes[V.local[t.dbox]].grown(nghost);
        const int n0 = g.len(0), n1 = g.len(1);
        for (int k = 0; k < t.n[2]; ++k)
            for (int j = 0; j < t.n[1]; ++j)
                for (int i = 0; i < t.n[0]; ++i) {
                    int di = t.dlo[0] + i, dj = t.dlo[1] + j, dk = t.dlo[2] + k;
                    int64_t v = -2;     // remote source
                    if (t.sbox >= 0) {
                        int gs = V.ext[t.sbox];
                        const Box& S = V.boxes[gs];
                        int64_t lin = ((int64_t)(dk + t.shift[2] - S.lo[2]) * S.len(1) + (dj + t.shift[1] - S.lo[1])) * S.len(0) + (di + t.shift[0] - S.lo[0]);
                        v = ((int64_t)gs << 40) | lin;
                    }
                    out[off[t.dbox] + ((int64_t)(dk - g.lo[2]) * n1 + (dj - g.lo[1])) * n0 + (di - g.lo[0])] = v;
                }
    }
    return PA_OK;
}

static const PaFaceRec* find_face(const pa_hier* h, int lev, int box, int face) {
    const Hier& H = h->H;
    if (lev < 0 || lev >= H.nlev || box < 0 || box >= (int)H.lev[lev].boxes.size()) return nullptr;
    int lb = H.lev[lev].g2l[box];
    if (lb < 0) return nullptr;
    for (long long r = H.faces.level_rec_begin[lev]; r < H.faces.level_rec_begin[lev + 1]; ++r)
        if (H.faces.recs[r].box == lb && H.faces.recs[r].face == face) return &H.faces.recs[r];
    return nullptr;
}
int64_t pa_debug_face_flags(pa_hier* h, int lev, int box, int face, uint16_t* out, int64_t out_len) {
    if (!h) return 0;
    const PaFaceRec* R = find_face(h, lev, box, face);
    if (!R) return 0;
    int64_t n = (int64_t)R->n1 * R->n2;
    if (out) {
        if (out_len < n) { fail(PA_ERR_ARG, "output buffer too small"); return -1; }
        std::memcpy(out, h->H.faces.flags.data() + R->start, (size_t)n * sizeof(uint16_t));
    }
    return n;
}
int pa_debug_face_coef(pa_hier* h, int lev, int box, int face, int* kind, int* nx, double coef[4]) {
    if (!h) return fail(PA_ERR_ARG, "null");
    const PaFaceRec* R = find_face(h, lev, box, face);
    if (!R) return fail(PA_ERR_ARG, "no record for this face");
    if (kind) *kind = R->kind;
    if (nx) *nx = R->nx;
    if (coef) for (int m = 0; m < 4; ++m) coef[m] = R->coef[m];
    return PA_OK;
}

int pa_debug_links(pa_hier* h, int lev, int box, int out[30]) {
    if (!h || !out || lev < 0 || lev >= h->H.nlev || box < 0 || box >= (int)h->H.lev[lev].boxes.size())
        return fail(PA_ERR_ARG, "pa_debug_links: bad argument");
    const Level& V = h->H.lev[lev];
    for (int f = 0; f < 6; ++f) {
        const Level::Link& K = V.link[box][f];
        out[5 * f] = K.nb;
        out[5 * f + 1] = K.nb >= 0 ? V.owner[K.nb] : -1;
        for (int d = 0; d < 3; ++d) out[5 * f + 2 + d] = K.nb >= 0 ? V.boxes[box].lo[d] + K.shift[d] - V.boxes[K.nb].lo[d] : 0;
    }
    return PA_OK;
}

int64_t pa_debug_selftest_math(int64_t n, uint64_t seed) {
    if (n < 1) { fail(PA_ERR_ARG, "pa_debug_selftest_math: n < 1"); return -1; }
    unsigned long long bad = 0;
    cudaError_t e = selftest_math((long long)n, (unsigned long long)seed, &bad, t_stream);
    if (e != cudaSuccess) { cuda_fail(e, "pa_debug_selftest_math"); return -1; }
    return (int64_t)bad;
}

int pa_debug_normal_math(void) { return stencil_tma_normal_math(); }
int pa_debug_curv_fused(pa_hier* h) {
    if (!h) return -1;
    if (ensure_device(h) != PA_OK) return -1;
    return h->curv_ok ? 1 : 0;
}
int64_t pa_debug_curv_fused_launches(void) { return g_fused_launches; }

int64_t pa_debug_exchange_ids(pa_hier* h, int which, int64_t* out, int64_t out_len) {
    if (!h) return 0;
    const std::vector<long long>& v = which ? h->H.xplan.recv_ids : h->H.xplan.send_ids;
    if (out) for (int64_t i = 0; i < (int64_t)v.size() && i < out_len; ++i) out[i] = v[i];
    return (int64_t)v.size();
}

// ------------------------------------------------------------------------------------------------ filterPlt path
// Filter::Filter(type, fgr) + set_*_weights (PelePhysics Source/Utility/Filter/Filter.H:56-111, Filter.cpp:3-404): ghost width
// and the 1-D weights.  The formulas and the Sagaut & Grohens (1999) ratio tables are data of the method; the arithmetic
// follows the reference expression by expression so that the weights agree to the last bit (same libm).
static int filter_weights_host(int type, int fgr, std::vector<double>& w) {
    auto box = [&](void) { const int ng = fgr / 2, n = 2 * ng + 1; w.assign(n, 1.0 / fgr); if (fgr > 1) { w[0] = 0.5 * w[0]; w[n - 1] = w[0]; } return ng; };
    auto box3 = [&](void) { w.assign(3, 0.0); w[0] = fgr * fgr / 24.0; w[1] = (12.0 - fgr * fgr) / 12.0; w[2] = w[0]; return 1; };
    auto gauss5 = [&](void) { const int f2 = fgr * fgr, f4 = f2 * f2; w.assign(5, 0.0); w[0] = (f4 - 4.0 * f2) / 1152.0; w[1] = (16.0 * f2 - f4) / 288.0;
                              w[2] = (f4 - 20.0 * f2 + 192.0) / 192.0; w[3] = w[1]; w[4] = w[0]; return 2; };
    static const double o3b[10] = {0.079, 0.274, 1.377, -2.375, -1.000, -0.779, -0.680, -0.627, -0.596, -0.575};
    static const double o3g[10] = {0.0763, 0.2527, 1.1160, -3.144, -1.102, -0.809, -0.696, -0.638, -0.604, -0.581};
    static const double o5b[10][2] = {{0.0886, -0.0169}, {0.3178, -0.0130}, {1.0237, 0.0368}, {2.4414, 0.5559}, {0.2949, 0.7096},
                                      {-0.5276, 0.4437}, {-0.6708, 0.3302}, {-0.7003, 0.2767}, {-0.7077, 0.2532}, {-0.6996, 0.2222}};
    static const double o5g[10][2] = {{0.0871, -0.0175}, {0.2596, -0.0021}, {0.4740, 0.0785}, {0.1036, 0.2611}, {-0.4252, 0.3007},
                                      {-0.6134, 0.2696}, {-0.6679, 0.2419}, {-0.6836, 0.2231}, {-0.6873, 0.2103}, {-0.6870, 0.2014}};
    switch (type) {
    case 1: return box();
    case 2: {
        const int ng = fgr / 2, n = 2 * ng + 1;
        w.assign(n, 0.0);
        const double gamma = 6.0, sigma = std::sqrt(1.0 / (2.0 * gamma)) * fgr;
        for (int i = 0; i < n; ++i) w[i] = 1.0 / (std::sqrt(2.0 * 3.1415926535897932384626433832795029) * sigma) * std::exp((-(i - ng) * (i - ng)) / (2 * sigma * sigma));
        double sum = 0.0;
        for (int i = 0; i < n; ++i) sum += w[i];
        for (int i = 0; i < n; ++i) w[i] /= sum;
        return ng;
    }
    case 3: case 7: return box3();
    case 4: {
        const int f2 = fgr * fgr, f4 = f2 * f2;
        w.assign(5, 0.0);
        w[0] = (3.0 * f4 - 20.0 * f2) / 5760.0; w[1] = (80.0 * f2 - 3.0 * f4) / 1440.0; w[2] = (3.0 * f4 - 100.0 * f2 + 960.0) / 960.0; w[3] = w[1]; w[4] = w[0];
        return 2;
    }
    case 5: case 9: {
        if (fgr < 1 || fgr > 10) return type == 5 ? box() : box3();
        const double ratio = (type == 5 ? o3b : o3g)[fgr - 1];
        w.assign(3, 0.0);
        w[0] = ratio / (1 + 2.0 * ratio); w[1] = 1.0 - 2.0 * w[0]; w[2] = w[0];
        return 1;
    }
    case 6: case 10: {
        if (fgr < 1 || fgr > 10) return type == 6 ? box() : gauss5();
        const double r1 = (type == 6 ? o5b : o5g)[fgr - 1][0], r2 = (type == 6 ? o5b : o5g)[fgr - 1][1];
        w.assign(5, 0.0);
        w[0] = r2 / (1 + 2.0 * r1 + 2.0 * r2); w[1] = r1 / r2 * w[0]; w[2] = 1.0 - 2.0 * w[0] - 2.0 * w[1]; w[3] = w[1]; w[4] = w[0];
        return 2;
    }
    case 8: return gauss5();
    default: w.assign(1, 1.0); return 0;
    }
}

int pa_filter_weights(int filter_type, int fgr, int* ngrow, double* weights, int cap) {
    if (fgr < 1) return fail(PA_ERR_ARG, "pa_filter_weights: filter-to-grid ratio must be >= 1");
    if ((filter_type == 1 || filter_type == 2) && fgr != 1 && fgr % 2) return fail(PA_ERR_ARG, "pa_filter_weights: the box / Gaussian filters need an even filter-to-grid ratio");
    std::vector<double> w;
    const int ng = filter_weights_host(filter_type, fgr, w);
    if (ngrow) *ngrow = ng;
    if (weights) {
        if ((int)w.size() > cap) return fail(PA_ERR_ARG, "pa_filter_weights: weight buffer too small");
        for (size_t i = 0; i < w.size(); ++i) weights[i] = w[i];
    }
    return (int)w.size();
}

int pa_boxes_max_size(int nboxes, const int* boxes, int max_grid_size, int* out_boxes, int cap) {
    if (nboxes < 0 || (nboxes && !boxes) || max_grid_size < 1) { fail(PA_ERR_ARG, "pa_boxes_max_size: bad arguments"); return PA_ERR_ARG; }
    std::vector<Box> out;
    box_max_size(nboxes, boxes, max_grid_size, out);
    if (out_boxes) {
        if ((int)out.size() > cap) { fail(PA_ERR_ARG, "pa_boxes_max_size: output buffer too small"); return PA_ERR_ARG; }
        for (size_t b = 0; b < out.size(); ++b)
            for (int d = 0; d < 3; ++d) { out_boxes[6 * b + d] = out[b].lo[d]; out_boxes[6 * b + 3 + d] = out[b].hi[d]; }
    }
    return (int)out.size();
}

// ---- FillPatch on several ranks ------------------------------------------------------------------------------------------
// Arguments every FillPatch entry shares; (lev, nghost, interp_type) names the fill and its exchange plan.
static int fp_check(const pa_field* f, int comp, int ncomp, int lev, int nghost, const std::string& who) {
    CHK(check_field(f, comp, ncomp, who.c_str()));
    const Hier& H = f->h->H;
    if (lev < 0 || lev >= H.nlev) return fail(PA_ERR_ARG, who + ": level out of range");
    if (nghost < 0 || nghost > f->ng) return fail(PA_ERR_ARG, who + ": the field has fewer ghost layers than asked for");
    if (H.is_per[0] || H.is_per[1] || H.is_per[2])
        return fail(PA_ERR_UNSUPPORTED, who + ": periodic directions are not served -- the reference tool's PltFileManager geometry is never periodic");
    return PA_OK;
}

// Host tables of the fill and their device copy.  The nesting verdict is taken over every box of the level, so on several
// ranks all of them fail here, before any communication, or none does.
static int fp_tables(pa_hier* h, int lev, int nghost, int interp_type, const FillPatchTable** T, pa_hier::FpDev** D, const std::string& who) {
    const int cgrow = interp_type == 1 ? 1 : 0;
    const FillPatchTable& X = h->H.fill_patch(lev, nghost, cgrow);
    if (!X.err.empty()) return fail(PA_ERR_ARG, who + ": " + X.err);
    std::array<int, 3> key{lev, nghost, cgrow};
    auto it = h->fp.find(key);
    if (it == h->fp.end()) {
        auto d = std::make_unique<pa_hier::FpDev>();
        CU(d->pieces.upload(X.pieces, t_stream));
        CU(d->copies.upload(X.copies, t_stream));
        CU(d->clamps.upload(X.clamps, t_stream));
        CU(d->pack.upload(X.pack, t_stream));
        CU(d->unpack.upload(X.unpack, t_stream));
        it = h->fp.emplace(key, std::move(d)).first;
    }
    *T = &X;
    *D = it->second.get();
    return PA_OK;
}

// send / recv slabs large enough for this plan; growing one must not free memory a queued pack or unpack still uses
static int fp_slabs(pa_hier* h, const FillPatchTable& T, int ncomp) {
    const int n = h->H.nranks;
    const size_t ns = (size_t)std::max<long long>(T.send_prefix[n] * ncomp, 1), nr = (size_t)std::max<long long>(T.recv_prefix[n] * ncomp, 1);
    if (h->fp_send.n < ns || h->fp_recv.n < nr) {
        CU(cudaStreamSynchronize(t_stream));
        CU(h->fp_send.reserve(ns));
        CU(h->fp_recv.reserve(nr));
    }
    return PA_OK;
}

// FabArray::FillPatchTwoLevels' communication (ParallelCopy of the coarse patches, FillBoundary of the fine level) as one
// slab exchange per fill: pa_fill_patch_pack -> transport (NCCL send/recv, pa_copy_async, ...) -> pa_fill_patch_mark_received
// -> pa_fill_patch.  On one rank the offsets are all zero and pack / mark do nothing.
int pa_fill_patch_exchange_buffers(pa_field* f, int ncomp, int lev, int nghost, int interp_type, double** send_slab, double** recv_slab,
                                   int64_t* send_offsets, int64_t* recv_offsets) {
    const std::string who = "pa_fill_patch_exchange_buffers";
    CHK(fp_check(f, 0, ncomp, lev, nghost, who));
    pa_hier* h = f->h;
    const int n = h->H.nranks;
    if (send_slab) *send_slab = nullptr;
    if (recv_slab) *recv_slab = nullptr;
    for (int p = 0; p <= n; ++p) {
        if (send_offsets) send_offsets[p] = 0;
        if (recv_offsets) recv_offsets[p] = 0;
    }
    if (n <= 1 || nghost == 0) return PA_OK;
    CHK(ensure_device(h));
    const FillPatchTable* T;
    pa_hier::FpDev* D;
    CHK(fp_tables(h, lev, nghost, interp_type, &T, &D, who));
    CHK(fp_slabs(h, *T, ncomp));
    if (send_slab) *send_slab = h->fp_send.p;
    if (recv_slab) *recv_slab = h->fp_recv.p;
    for (int p = 0; p <= n; ++p) {
        if (send_offsets) send_offsets[p] = T->send_prefix[p] * ncomp;
        if (recv_offsets) recv_offsets[p] = T->recv_prefix[p] * ncomp;
    }
    return PA_OK;
}

int pa_fill_patch_pack(pa_field* f, int comp, int ncomp, int lev, int nghost, int interp_type) {
    const std::string who = "pa_fill_patch_pack";
    CHK(fp_check(f, comp, ncomp, lev, nghost, who));
    pa_hier* h = f->h;
    h->fp_mark = pa_hier::FpMark();                  // the transport that follows overwrites the recv slab
    if (h->H.nranks <= 1 || nghost == 0) return PA_OK;
    CHK(ensure_device(h));
    const FillPatchTable* T;
    pa_hier::FpDev* D;
    CHK(fp_tables(h, lev, nghost, interp_type, &T, &D, who));
    CHK(fp_slabs(h, *T, ncomp));
    if (T->npack == 0) return PA_OK;
    GridArgs ga;
    CHK(grid_args_inplace(f, comp, ga));
    CU(launch_exchange_pack(D->pack.p, 0, (long long)T->pack.size(), 0, T->npack, ga, ncomp, h->fp_send.p, t_stream));
    return PA_OK;
}

int pa_fill_patch_mark_received(pa_field* f, int comp, int ncomp, int lev, int nghost, int interp_type) {
    CHK(fp_check(f, comp, ncomp, lev, nghost, "pa_fill_patch_mark_received"));
    pa_hier* h = f->h;
    if (h->H.nranks <= 1) return PA_OK;
    pa_hier::FpMark m;
    m.f = f; m.comp = comp; m.ncomp = ncomp; m.lev = lev; m.ng = nghost; m.cgrow = interp_type == 1 ? 1 : 0;
    h->fp_mark = m;
    return PA_OK;
}

int64_t pa_debug_fill_patch_exchange_ids(pa_hier* h, int lev, int nghost, int interp_type, int which, int64_t* out, int64_t out_len) {
    if (!h || lev < 0 || lev >= h->H.nlev || nghost < 0) { fail(PA_ERR_ARG, "pa_debug_fill_patch_exchange_ids: bad argument"); return PA_ERR_ARG; }
    const FillPatchTable& T = h->H.fill_patch(lev, nghost, interp_type == 1 ? 1 : 0);
    if (!T.err.empty()) { fail(PA_ERR_ARG, "pa_debug_fill_patch_exchange_ids: " + T.err); return PA_ERR_ARG; }
    const std::vector<long long>& v = which ? T.recv_ids : T.send_ids;
    if (out) for (int64_t i = 0; i < (int64_t)v.size() && i < out_len; ++i) out[i] = v[i];
    return (int64_t)v.size();
}

int pa_fill_patch(pa_field* f, int comp, int ncomp, int lev, int nghost, int interp_type) {
    CHK(fp_check(f, comp, ncomp, lev, nghost, "pa_fill_patch"));
    pa_hier* h = f->h;
    Hier& H = h->H;
    CHK(ensure_device(h));
    if (nghost == 0) return PA_OK;
    const int cgrow = interp_type == 1 ? 1 : 0;
    const FillPatchTable* Tp;
    pa_hier::FpDev* Dp;
    CHK(fp_tables(h, lev, nghost, interp_type, &Tp, &Dp, "pa_fill_patch"));
    const FillPatchTable& T = *Tp;
    const double* recv = nullptr;
    if (T.nunpack > 0) {
        const pa_hier::FpMark& m = h->fp_mark;
        if (m.f != f || m.comp != comp || m.ncomp != ncomp || m.lev != lev || m.ng != nghost || m.cgrow != cgrow)
            return fail(PA_ERR_ARG, "pa_fill_patch: this rank receives cells for the fill, but the recv slab does not hold them: exchange this "
                                    "(field, comp, ncomp, lev, nghost, interp_type) first (pa_fill_patch_pack -> transport -> pa_fill_patch_mark_received)");
        recv = h->fp_recv.p;
    }
    int err = PA_OK;
    const PaLayDev* lay = dev_layout(h, lev, f->ng, &err);
    if (!lay) return err;
    double* base = f->slab[lev] + (long long)comp * f->cs[lev];
    const Level& V = H.lev[lev];
    // 1. same-level valid data into every ghost cell another box of the level covers (`nghost` layers, edges and corners).
    //    The tags are in index space and the layout is passed separately, so the table of the level's own width serves a
    //    field that carries more layers (the widest level decides the field's ghost width).
    {
        auto key = std::make_pair(lev, nghost);
        const HaloTable& T = H.halo_full(lev, nghost);
        auto it = h->halo_full.find(key);
        if (it == h->halo_full.end()) {
            auto buf = std::make_unique<DevBuf<PaHaloTag>>();
            CU(buf->upload(T.tags, t_stream));
            it = h->halo_full.emplace(key, std::move(buf)).first;
        }
        // slices per tag: enough blocks for the device when the level has few, large tags (128^3 boxes: 65 k cells per face tag)
        const long long per_tag = T.tags.empty() ? 0 : T.ncells / (long long)T.tags.size();
        const int slices = (int)std::min<long long>(16, std::max<long long>(1, per_tag / 2048));
        CU(launch_halo_blocks(it->second->p, (int)T.tags.size(), slices, h->lev[lev]->boxes.p, lay, base, f->cs[lev], ncomp, t_stream));
    }
    // 2. the rest of the in-domain ghost cells from the next coarser level, 3. the out-of-domain ones by extrapolation.
    //    Several ranks: the unpack (cells of other ranks into ghost cells and coarse patches) joins 1. and 2. before the
    //    interpolation reads the patches; the clamp reads in-domain ghost cells, so it comes last.
    const pa_hier::FpDev* D = Dp;
    if (T.nfine > 0) {
        const size_t need = (size_t)T.ncrse * ncomp;
        if (h->fp_scratch.n < need) {
            CU(cudaStreamSynchronize(t_stream));          // an earlier fill may still read the buffer this replaces
            CU(h->fp_scratch.reserve(need));
        }
        if (T.ncopy > 0) {                                // several ranks: the coarse boxes of a patch may all be remote
            const PaLayDev* clay = dev_layout(h, lev - 1, f->ng, &err);
            if (!clay) return err;
            const double* cbase = f->slab[lev - 1] + (long long)comp * f->cs[lev - 1];
            CU(launch_fp_gather(D->copies.p, (int)T.copies.size(), T.ncopy, D->pieces.p, h->lev[lev - 1]->boxes.p, clay, cbase,
                                f->cs[lev - 1], ncomp, h->fp_scratch.p, T.ncrse, t_stream));
        }
    }
    CU(launch_fp_unpack(D->unpack.p, (int)T.unpack.size(), T.nunpack, recv, D->pieces.p, h->fp_scratch.p, T.ncrse, h->lev[lev]->boxes.p, lay,
                        base, f->cs[lev], ncomp, t_stream));
    if (T.nfine > 0) {
        const Level& Cv = H.lev[lev - 1];
        CU(launch_fp_interp(interp_type == 1, D->pieces.p, (int)T.pieces.size(), T.nfine, h->fp_scratch.p, T.ncrse, Cv.dom.lo, Cv.dom.hi,
                            V.ratio, h->lev[lev]->boxes.p, lay, base, f->cs[lev], ncomp, t_stream));
    }
    CU(launch_fp_clamp(D->clamps.p, (int)T.clamps.size(), T.nclamp, V.dom.lo, V.dom.hi, nghost, h->lev[lev]->boxes.p, lay, base,
                       f->cs[lev], ncomp, t_stream));
    return PA_OK;
}

int pa_filter(pa_field* in, int comp_in, pa_field* out, int comp_out, int ncomp, int lev, int filter_type, int fgr) {
    CHK(check_field(in, comp_in, ncomp, "pa_filter (in)"));
    CHK(check_field(out, comp_out, ncomp, "pa_filter (out)"));
    if (in->h != out->h) return fail(PA_ERR_ARG, "pa_filter: fields of different hierarchies");
    if (in == out) return fail(PA_ERR_ARG, "pa_filter: in and out must be different fields");
    pa_hier* h = in->h;
    Hier& H = h->H;
    if (lev < 0 || lev >= H.nlev) return fail(PA_ERR_ARG, "pa_filter: level out of range");
    std::vector<double> w;
    {
        const int rc = pa_filter_weights(filter_type, fgr, nullptr, nullptr, 0);
        if (rc < 0) return rc;
    }
    const int g = filter_weights_host(filter_type, fgr, w);
    if (g > in->ng) return fail(PA_ERR_ARG, "pa_filter: the input field has fewer ghost layers than the filter needs");
    CHK(ensure_device(h));
    const Level& V = H.lev[lev];
    const int nb = (int)V.local.size();
    if (nb == 0) return PA_OK;
    int err = PA_OK;
    const PaLayDev* lin = dev_layout(h, lev, in->ng, &err);
    if (!lin) return err;
    const PaLayDev* lout = dev_layout(h, lev, out->ng, &err);
    if (!lout) return err;
    auto pit = h->filter_prefix.find(lev);
    if (pit == h->filter_prefix.end()) {
        std::vector<long long> pre(nb + 1, 0);
        for (int b = 0; b < nb; ++b) {
            const Box& B = V.boxes[V.local[b]];
            pre[b + 1] = pre[b] + (long long)((B.len(0) + 3) / 4) * ((B.len(1) + 1) / 2) * B.len(2);   // blocks of 4 x 2 cells
        }
        auto buf = std::make_unique<DevBuf<long long>>();
        CU(buf->upload(pre, t_stream));
        h->filter_nwork[lev] = pre[nb];
        pit = h->filter_prefix.emplace(lev, std::move(buf)).first;
    }
    // weight products in the reference's order: ((w[l] * w[m]) * w[n]), n slowest
    const int W = 2 * g + 1;
    std::vector<double> w3((size_t)W * W * W);
    for (int n = 0; n < W; ++n)
        for (int m = 0; m < W; ++m)
            for (int l = 0; l < W; ++l) w3[((size_t)n * W + m) * W + l] = (w[l] * w[m]) * w[n];
    if (h->filter_w3.n < w3.size()) {
        CU(cudaStreamSynchronize(t_stream));
        CU(h->filter_w3.reserve(std::max<size_t>(w3.size(), 729)));
    }
    // pageable source: the runtime stages the bytes before returning, so w3 may go out of scope
    CU(cudaMemcpyAsync(h->filter_w3.p, w3.data(), w3.size() * sizeof(double), cudaMemcpyHostToDevice, t_stream));
    CU(launch_filter(g, h->lev[lev]->boxes.p, lin, lout, nb, pit->second->p, h->filter_nwork[lev], in->slab[lev] + (long long)comp_in * in->cs[lev],
                     in->cs[lev], out->slab[lev] + (long long)comp_out * out->cs[lev], out->cs[lev], ncomp, h->filter_w3.p, t_stream));
    return PA_OK;
}

// Measured FP64 rate of this GPU for separate multiplies and adds (the filter's instruction mix, no FMA): Gop/s.
int pa_debug_fp64_rate(double* gops) {
    if (!gops) return fail(PA_ERR_ARG, "pa_debug_fp64_rate: null output");
#ifdef PA_HOST_EMULATION
    return fail(PA_ERR_UNSUPPORTED, "pa_debug_fp64_rate: a timing measurement, GPU only");
#else
    cudaError_t esm = cudaSuccess;
    const int nsm = stencil_num_sms(&esm);
    if (esm != cudaSuccess) return cuda_fail(esm, "device query");
    const int blocks = nsm * 8, threads = 256, iters = 4096;
    double* buf = nullptr;
    CU(dev_alloc((void**)&buf, (size_t)blocks * threads * sizeof(double)));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaError_t e = launch_fp64_rate(buf, blocks, threads, 64, t_stream);        // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 3 && e == cudaSuccess; ++rep) {
        cudaEventRecord(e0, t_stream);
        e = launch_fp64_rate(buf, blocks, threads, iters, t_stream);
        cudaEventRecord(e1, t_stream);
        if (e == cudaSuccess) e = cudaEventSynchronize(e1);
        float ms = 0.f;
        if (e == cudaSuccess) { cudaEventElapsedTime(&ms, e0, e1); best = std::min(best, ms); }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    dev_free(buf);
    if (e != cudaSuccess) return cuda_fail(e, "pa_debug_fp64_rate");
    *gops = (double)blocks * threads * iters * 16.0 / (best * 1e-3) / 1e9;
    return PA_OK;
#endif
}

}  // extern "C"
