// multi_gpu.hpp -- the grad, curvature and filterPlt tools on several GPUs of one node from ONE process: one host thread per
// GPU, no MPI, no NCCL.
//
// What an MPI build of the reference does rank by rank (boxes distributed by DistributionMapping, ghost cells through
// FillBoundary / ParallelCopy, one Cell_D file per rank) is done here thread by thread: thread r owns GPU r and the boxes the
// SFC distribution gives rank r, reads only those from disk, moves the ghost sources owned by other threads as packed slabs
// with device-to-device copies (pa_copy_async), runs the tool's C-ABI calls, and writes its own boxes to Level_l/Cell_D_<r>;
// thread 0 writes Header and Cell_H.  Barriers between threads stand where the reference has MPI synchronisation: before
// anyone reads a peer's slab, and before anyone frees a slab a peer may still read.
// grad and curvature have two transports (key transport=peer|slab): with peer links (the default) every thread also maps the
// other threads' level slabs (pa_field_map_peer_ptr) and the stencil kernels read cross-GPU neighbour faces and coarse cells in
// place over NVLink, so only the ragged remainder travels in the slabs; with transport=slab no field slab is mapped and every
// ghost source of another thread travels in the slabs (the width-1 exchange plan of hier.cpp: build_exchange), as filterPlt's
// FillPatch sources always do.  Every transport enables peer access between the GPUs: it lets the copy engines move the
// pa_copy_async copies GPU to GPU directly instead of through host memory.
#pragma once
#include <condition_variable>
#include <cstdio>
#include <mutex>
#include <thread>

#include "tool_common.hpp"

struct ThreadBarrier {
    explicit ThreadBarrier(int n) : n_(n) {}
    void wait() {
        std::unique_lock<std::mutex> lk(mu_);
        const int gen = gen_;
        if (++count_ == n_) { count_ = 0; ++gen_; cv_.notify_all(); }
        else cv_.wait(lk, [&] { return gen_ != gen; });
    }
private:
    std::mutex mu_;
    std::condition_variable cv_;
    int n_, count_ = 0, gen_ = 0;
};

struct MultiShared {
    explicit MultiShared(int n) : n(n), bar(n), slab(n), send(n, nullptr), soff(n), mapped(n, 0), received(n, 0) {}
    int n;
    ThreadBarrier bar;
    std::mutex mu;
    std::vector<std::vector<const double*>> slab;      // [rank][level] (grad) / [rank][field * nlev + level]: level slabs, published for the peers
    std::vector<double*> send;                         // [rank]: send slab
    std::vector<std::vector<int64_t>> soff;            // [rank][peer .. ]: offsets into it
    std::vector<pltio::FabRecord> records;             // what every thread wrote
    long long launches = 0;
    std::vector<long long> mapped;                     // [rank]: peer level slabs mapped (pa_field_map_peer_ptr calls)
    std::vector<long long> received;                   // [rank]: doubles received through the slabs over the whole run
};

// verbose=1: what crossed between the GPUs, one line (the transport is visible in it: no slab is mapped with transport=slab)
inline void print_transport_report(const MultiShared& M, bool peer) {
    std::cout << "[b200] transport=" << (peer ? "peer" : "slab") << ": peer slabs mapped per GPU";
    for (long long v : M.mapped) std::cout << " " << v;
    std::cout << "; doubles received through slabs per GPU";
    for (long long v : M.received) std::cout << " " << v;
    std::cout << std::endl;
}

// every thread publishes the level slabs of its fields, then maps everyone else's (collective: all threads call it with the
// same number of fields in the same order)
inline void map_all_peers(int r, MultiShared& M, int nlev, const std::vector<pa_field*>& fields) {
    M.slab[r].assign(fields.size() * nlev, nullptr);
    for (size_t f = 0; f < fields.size(); ++f)
        for (int l = 0; l < nlev; ++l) check(pa_field_slab(fields[f], l, &M.slab[r][f * nlev + l]), "pa_field_slab");
    M.bar.wait();
    for (int p = 0; p < M.n; ++p)
        if (p != r)
            for (size_t f = 0; f < fields.size(); ++f)
                for (int l = 0; l < nlev; ++l) {
                    check(pa_field_map_peer_ptr(fields[f], l, p, M.slab[p][f * nlev + l]), "pa_field_map_peer_ptr");
                    ++M.mapped[r];
                }
    M.bar.wait();
}

// The cross-rank step in front of a ghost fill (collective): what the neighbour links do not cover -- ragged same-level
// neighbours, coarse cells of coarse-fine faces owned by another rank -- moves as packed slabs.  Its first barrier is also the
// ordering point peer links need: every rank has finished (pa_sync) whatever wrote the data its peers are about to read.
inline void exchange_slabs(int r, MultiShared& M, pa_field* f, int comp, int ncomp) {
    const int n = M.n;
    double *send = nullptr, *recv = nullptr;
    std::vector<int64_t> so(n + 1), ro(n + 1);
    check(pa_exchange_buffers(f, ncomp, &send, &recv, so.data(), ro.data()), "pa_exchange_buffers");
    check(pa_exchange_pack(f, comp, ncomp), "pa_exchange_pack");
    check(pa_sync(), "pa_sync");
    M.send[r] = send;
    M.soff[r] = so;
    M.bar.wait();
    for (int p = 0; p < n; ++p) {
        if (p == r) continue;
        const int64_t cnt = ro[p + 1] - ro[p];
        if (cnt != M.soff[p][r + 1] - M.soff[p][r]) pa_abort("multi-GPU exchange plan: send / recv counts disagree");
        if (cnt > 0) check(pa_copy_async(recv + ro[p], M.send[p] + M.soff[p][r], cnt), "pa_copy_async");
    }
    M.received[r] += ro[n];
    check(pa_exchange_mark_received(f, comp, ncomp), "pa_exchange_mark_received");
    check(pa_sync(), "pa_sync");
    M.bar.wait();                                      // the send slabs may be repacked from here on
}

struct GradJob {
    std::string infile, outfile;
    const pltio::Header* H;
    int Nlev;
    std::vector<std::string> gvars, aux, names;
    std::vector<int> is_per;
    int bck[3];
    bool peer = true;                                  // transport=peer (peer links + slabs) or slab (packed slabs only)
    bool verbose = false;                              // print_transport_report after the run
    std::vector<std::vector<int>> owner;               // [level][box] -> rank
};

// the hierarchy flags of a grad / curvature rank for its transport
inline unsigned transport_flags(bool peer) { return peer ? PA_HIER_PEER_LINKS : 0u; }

inline void grad_rank(int r, MultiShared& M, const GradJob& J) {
    const pltio::Header& H = *J.H;
    const int n = M.n, Nlev = J.Nlev, nv = (int)J.gvars.size(), nAux = (int)J.aux.size();
    const int nIn = nv + nAux, nOut = nIn + 4 * nv;
    check(pa_init(r), "pa_init");
    for (int p = 0; p < n; ++p) if (p != r) check(pa_enable_peer_access(p), "pa_enable_peer_access");
    HierInput hi;
    make_level_descs(H, Nlev, hi);
    std::vector<std::vector<int>> own(Nlev), mine(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        own[l] = J.owner[l];
        hi.lv[l].owner = own[l].data();
        for (int b = 0; b < (int)own[l].size(); ++b) if (own[l][b] == r) mine[l].push_back(b);
    }
    pa_hier* h = nullptr;
    check(pa_hier_create2(&h, Nlev, hi.lv.data(), J.is_per.data(), J.bck, r, n, transport_flags(J.peer)), "pa_hier_create2");
    pa_field *fin = nullptr, *fout = nullptr;
    check(pa_field_alloc(h, nv, 1, &fin), "pa_field_alloc");
    check(pa_field_alloc(h, 4 * nv, 0, &fout), "pa_field_alloc");

    // this rank's boxes: gradient variables to the device, pass-through variables stay on the host
    std::vector<PinnedLevel> buf(Nlev);
    std::vector<long long> ncell(Nlev, 0);
    for (int l = 0; l < Nlev; ++l) {
        for (int b : mine[l]) ncell[l] += H.levels[l].boxes[b].npts();
        buf[l].alloc(std::max<long long>(ncell[l], 1), nOut);
        if (mine[l].empty()) continue;
        for (int v = 0; v < nv; ++v) {
            pltio::read_boxes_comp(J.infile, H, l, H.comp(J.gvars[v]), mine[l], buf[l].comp(v));
            check(pa_field_upload_level(fin, l, v, buf[l].comp(v)), "upload");
        }
        for (int a = 0; a < nAux; ++a) pltio::read_boxes_comp(J.infile, H, l, H.comp(J.aux[a]), mine[l], buf[l].comp(nv + a));
    }
    check(pa_sync(), "pa_sync");

    if (J.peer) map_all_peers(r, M, Nlev, {fin});
    exchange_slabs(r, M, fin, 0, nv);

    check(pa_grad(fin, 0, nv, fout, 0), "pa_grad");
    for (int l = 0; l < Nlev; ++l)
        if (!mine[l].empty())
            for (int c = 0; c < 4 * nv; ++c) check(pa_field_download_level(fout, l, c, buf[l].comp(nIn + c)), "download");
    check(pa_sync(), "pa_sync");
    M.bar.wait();                                                     // nobody frees a slab (or send slab) a peer may still be reading

    char fn[32];
    std::snprintf(fn, sizeof fn, "Cell_D_%05d", r);
    std::vector<pltio::FabRecord> recs;
    for (int l = 0; l < Nlev; ++l) {
        std::vector<const double*> data;
        for (int c = 0; c < nOut; ++c) data.push_back(buf[l].comp(c));
        auto w = pltio::write_fab_file(J.outfile, H, l, fn, mine[l], data);
        recs.insert(recs.end(), w.begin(), w.end());
    }
    {
        std::lock_guard<std::mutex> lk(M.mu);
        M.records.insert(M.records.end(), recs.begin(), recs.end());
        M.launches = pa_kernel_launches();
    }
    pa_field_free(fin); pa_field_free(fout); pa_hier_destroy(h);
    M.bar.wait();
}

inline std::vector<std::vector<int>> sfc_owners(const pltio::Header& H, int Nlev, int ngpus) {
    std::vector<std::vector<int>> owner(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        std::vector<int> bx;
        for (auto& b : H.levels[l].boxes) { for (int d = 0; d < 3; ++d) bx.push_back(b.lo[d]); for (int d = 0; d < 3; ++d) bx.push_back(b.hi[d]); }
        owner[l].resize(H.levels[l].boxes.size());
        check(pa_sfc_distribute((int)H.levels[l].boxes.size(), bx.data(), ngpus, owner[l].data()), "pa_sfc_distribute");
    }
    return owner;
}

// returns after the output plotfile is complete
inline void run_grad_multi(int ngpus, GradJob& J) {
    const pltio::Header& H = *J.H;
    J.owner = sfc_owners(H, J.Nlev, ngpus);
    try { pltio::create_plotfile_dirs(J.outfile, J.Nlev); } catch (std::exception& e) { pa_abort(e.what()); }
    MultiShared M(ngpus);
    std::vector<std::thread> th;
    for (int r = 0; r < ngpus; ++r) th.emplace_back([&, r] {
        try { grad_rank(r, M, J); } catch (std::exception& e) { pa_abort(e.what()); }
    });
    for (auto& t : th) t.join();
    if (J.verbose) print_transport_report(M, J.peer);
    std::vector<int> rr(std::max(J.Nlev - 1, 0), 2);              // the reference hard-codes refRatios = 2 (grad.cpp:255)
    pltio::Header meta = H;
    meta.time = 0.0;                                               // WriteMultiLevelPlotfile(..., 0.0, ...) (grad.cpp:256)
    try { pltio::write_metadata(J.outfile, meta, J.names, J.Nlev, M.records, rr); } catch (std::exception& e) { pa_abort(e.what()); }
}

// ---- curvature: the steps of pa_curvature_steps with the cross-rank step each one needs in front of it ---------------------
struct CurvJob {
    std::string infile, outfile;
    const pltio::Header* H;
    int Nlev;
    std::vector<std::string> inNames, velNames, names;   // pass-through inputs (progress variable first), velocities, output names
    bool need_vel;
    pa_curv_opts o;
    std::vector<int> slot;                               // library result component -> output slot
    std::vector<int> zero_slots;                         // output slots nothing writes (the reference leaves them uninitialised)
    int nCompOut;
    std::vector<int> is_per;
    int bck[3];
    bool peer = true;                                    // as GradJob::peer
    bool verbose = false;
    std::vector<std::vector<int>> owner;
};

inline void curv_rank(int r, MultiShared& M, const CurvJob& J) {
    const pltio::Header& H = *J.H;
    const int n = M.n, Nlev = J.Nlev, nCompIn = (int)J.inNames.size();
    check(pa_init(r), "pa_init");
    for (int p = 0; p < n; ++p) if (p != r) check(pa_enable_peer_access(p), "pa_enable_peer_access");
    HierInput hi;
    make_level_descs(H, Nlev, hi);
    std::vector<std::vector<int>> own(Nlev), mine(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        own[l] = J.owner[l];
        hi.lv[l].owner = own[l].data();
        for (int b = 0; b < (int)own[l].size(); ++b) if (own[l][b] == r) mine[l].push_back(b);
    }
    pa_hier* h = nullptr;
    check(pa_hier_create2(&h, Nlev, hi.lv.data(), J.is_per.data(), J.bck, r, n, transport_flags(J.peer)), "pa_hier_create2");
    const int nres = pa_curvature_num_outputs(&J.o);
    pa_field *st = nullptr, *res = nullptr, *scratch = nullptr;
    check(pa_field_alloc(h, J.need_vel ? 4 : 1, 1, &st), "pa_field_alloc");
    check(pa_field_alloc(h, nres, 1, &res), "pa_field_alloc");
    if (J.o.do_gauss) check(pa_curvature_scratch(h, 0, &scratch), "pa_curvature_scratch");

    std::vector<PinnedLevel> buf(Nlev), velbuf(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        long long nc = 0;
        for (int b : mine[l]) nc += H.levels[l].boxes[b].npts();
        buf[l].alloc(std::max<long long>(nc, 1), J.nCompOut);
        buf[l].ncells = nc;
        if (J.need_vel) { velbuf[l].alloc(std::max<long long>(nc, 1), 3); velbuf[l].ncells = nc; }
        if (mine[l].empty()) continue;
        for (int c = 0; c < nCompIn; ++c) pltio::read_boxes_comp(J.infile, H, l, H.comp(J.inNames[c]), mine[l], buf[l].p + (long long)c * std::max<long long>(nc, 1));
        check(pa_field_upload_level(st, l, 0, buf[l].p), "upload");
        if (J.need_vel)
            for (int d = 0; d < 3; ++d) {
                double* v = velbuf[l].p + (long long)d * std::max<long long>(nc, 1);
                pltio::read_boxes_comp(J.infile, H, l, H.comp(J.velNames[d]), mine[l], v);
                check(pa_field_upload_level(st, l, 1 + d, v), "upload");
            }
    }
    check(pa_sync(), "pa_sync");
    std::vector<pa_field*> fields{st, res};
    if (scratch) fields.push_back(scratch);
    if (J.peer) map_all_peers(r, M, Nlev, fields);

    auto step = [&](int steps, int lo, int hi) { check(pa_curvature_steps(st, 0, 1, &J.o, res, 0, steps, lo, hi), "pa_curvature_steps"); };
    exchange_slabs(r, M, st, 0, 1);
    step(PA_CURV_PASS1, -1, -1);
    if (J.o.do_threshold) {
        for (int l = 0; l < Nlev; ++l) {
            exchange_slabs(r, M, res, 2, 3);
            step(PA_CURV_DIV, l, l);
            // the clip zeroes n(l) in place; with peer links every rank's DIV(l) reads its peers' UNCLIPPED n(l) over the links
            // first (curvature.cpp:487-567: FillBoundary of n precedes the clip).  With transport=slab the peers' cells of n(l)
            // were copied inside exchange_slabs, which ends in a barrier: nothing reads n(l) in place.
            if (J.peer) {
                check(pa_sync(), "pa_sync");
                M.bar.wait();
            }
            step(PA_CURV_CLIP, l, l);
        }
    } else {
        exchange_slabs(r, M, res, 2, 3);
        step(PA_CURV_DIV, -1, -1);
    }
    if (J.o.do_gauss) { exchange_slabs(r, M, scratch, 0, 3); step(PA_CURV_GAUSS, -1, -1); }
    if (J.o.do_strain) { exchange_slabs(r, M, st, 1, 3); step(PA_CURV_STRAIN, -1, -1); }
    if (J.o.do_velnormal) step(PA_CURV_VELN, -1, -1);

    for (int l = 0; l < Nlev; ++l) {
        const long long stride = std::max<long long>(buf[l].ncells, 1);
        for (int z : J.zero_slots) std::fill(buf[l].p + z * stride, buf[l].p + z * stride + buf[l].ncells, 0.0);
        if (!mine[l].empty())
            for (int c = 0; c < nres; ++c) check(pa_field_download_level(res, l, c, buf[l].p + (long long)J.slot[c] * stride), "download");
    }
    check(pa_sync(), "pa_sync");
    M.bar.wait();                                                     // nobody frees a slab a peer may still be reading

    char fn[32];
    std::snprintf(fn, sizeof fn, "Cell_D_%05d", r);
    std::vector<pltio::FabRecord> recs;
    for (int l = 0; l < Nlev; ++l) {
        const long long stride = std::max<long long>(buf[l].ncells, 1);
        std::vector<const double*> data;
        for (int c = 0; c < J.nCompOut; ++c) data.push_back(buf[l].p + (long long)c * stride);
        auto w = pltio::write_fab_file(J.outfile, H, l, fn, mine[l], data);
        recs.insert(recs.end(), w.begin(), w.end());
    }
    {
        std::lock_guard<std::mutex> lk(M.mu);
        M.records.insert(M.records.end(), recs.begin(), recs.end());
    }
    pa_field_free(st); pa_field_free(res); pa_hier_destroy(h);
    M.bar.wait();
}

inline void run_curv_multi(int ngpus, CurvJob& J) {
    const pltio::Header& H = *J.H;
    J.owner = sfc_owners(H, J.Nlev, ngpus);
    try { pltio::create_plotfile_dirs(J.outfile, J.Nlev); } catch (std::exception& e) { pa_abort(e.what()); }
    MultiShared M(ngpus);
    std::vector<std::thread> th;
    for (int r = 0; r < ngpus; ++r) th.emplace_back([&, r] {
        try { curv_rank(r, M, J); } catch (std::exception& e) { pa_abort(e.what()); }
    });
    for (auto& t : th) t.join();
    if (J.verbose) print_transport_report(M, J.peer);
    std::vector<int> rr(std::max(J.Nlev - 1, 0), 2);              // curvature.cpp:842
    pltio::Header meta = H;
    meta.time = 0.0;
    try { pltio::write_metadata(J.outfile, meta, J.names, J.Nlev, M.records, rr); } catch (std::exception& e) { pa_abort(e.what()); }
}

// ---- filterPlt: boxes of every level spread over the threads, FillPatch sources of other ranks moved as packed slabs -----
// The exchange in front of pa_fill_patch(lev): pack -> device-to-device copies of each peer's segment (pa_copy_async, as
// exchange_slabs) -> mark.  Collective; the filterPlt hierarchy has no peer links, so nothing is read in place.
inline void exchange_fill_patch(int r, MultiShared& M, pa_field* f, int ncomp, int lev, int nghost, int interp_type) {
    const int n = M.n;
    double *send = nullptr, *recv = nullptr;
    std::vector<int64_t> so(n + 1), ro(n + 1);
    check(pa_fill_patch_exchange_buffers(f, ncomp, lev, nghost, interp_type, &send, &recv, so.data(), ro.data()), "pa_fill_patch_exchange_buffers");
    check(pa_fill_patch_pack(f, 0, ncomp, lev, nghost, interp_type), "pa_fill_patch_pack");
    check(pa_sync(), "pa_sync");
    M.send[r] = send;
    M.soff[r] = so;
    M.bar.wait();
    for (int p = 0; p < n; ++p) {
        if (p == r) continue;
        const int64_t cnt = ro[p + 1] - ro[p];
        if (cnt != M.soff[p][r + 1] - M.soff[p][r]) pa_abort("multi-GPU FillPatch plan: send / recv counts disagree");
        if (cnt > 0) check(pa_copy_async(recv + ro[p], M.send[p] + M.soff[p][r], cnt), "pa_copy_async");
    }
    check(pa_fill_patch_mark_received(f, 0, ncomp, lev, nghost, interp_type), "pa_fill_patch_mark_received");
    check(pa_sync(), "pa_sync");
    M.bar.wait();                                      // the send slabs may be repacked from here on
}

struct FilterJob {
    std::string infile, outfile;
    const pltio::Header* H;                            // the plotfile
    const pltio::Header* meta;                         // its grids re-chopped to max_grid_size (the output's boxes)
    std::vector<std::vector<int>> parent;              // [level][output box] -> the plotfile box it was cut from
    int Nlev, filter_type, interp_type, ngmax;
    std::vector<int> fgr, ngrow;
    std::vector<std::string> names;
    std::vector<std::vector<int>> owner;               // [level][output box] -> rank
};

inline void filter_rank(int r, MultiShared& M, const FilterJob& J) {
    const pltio::Header& H = *J.H;
    const pltio::Header& meta = *J.meta;
    const int n = M.n, Nlev = J.Nlev, ncomp = (int)J.names.size();
    const bool talk = r == 0;                          // the tool's progress messages, once
    check(pa_init(r), "pa_init");
    for (int p = 0; p < n; ++p) if (p != r) check(pa_enable_peer_access(p), "pa_enable_peer_access");
    HierInput hi;
    make_level_descs(meta, Nlev, hi);
    std::vector<std::vector<int>> own(Nlev), mine(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        own[l] = J.owner[l];
        hi.lv[l].owner = own[l].data();
        for (int b = 0; b < (int)own[l].size(); ++b) if (own[l][b] == r) mine[l].push_back(b);
    }
    const int no_per[3] = {0, 0, 0}, bck[3] = {PA_BC_NEUMANN, PA_BC_NEUMANN, PA_BC_NEUMANN};
    pa_hier* h = nullptr;
    check(pa_hier_create2(&h, Nlev, hi.lv.data(), no_per, bck, r, n, PA_HIER_FILTER_ONLY), "pa_hier_create2");
    pa_field *fin = nullptr, *fout = nullptr;
    check(pa_field_alloc(h, ncomp, J.ngmax, &fin), "pa_field_alloc");
    check(pa_field_alloc(h, ncomp, 0, &fout), "pa_field_alloc");

    // this rank's output boxes, cut from the plotfile boxes that contain them (only those are read)
    if (talk) std::cout << "Reading data..." << std::endl;
    std::vector<PinnedLevel> buf(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        if (talk) std::cout << "on level " << l << std::endl;
        long long nc = 0;
        for (int b : mine[l]) nc += meta.levels[l].boxes[b].npts();
        buf[l].alloc(std::max<long long>(nc, 1), ncomp);
        buf[l].ncells = nc;
        if (mine[l].empty()) continue;
        std::vector<double> tmp;
        for (int v = 0; v < ncomp; ++v) {
            double* dst = buf[l].comp(v);
            for (size_t i = 0; i < mine[l].size();) {
                const int pb = J.parent[l][mine[l][i]];
                const pltio::BoxI& B = H.levels[l].boxes[pb];
                tmp.resize((size_t)B.npts());
                pltio::read_boxes_comp(J.infile, H, l, H.comp(J.names[v]), {pb}, tmp.data());
                const long long nx = B.hi[0] - B.lo[0] + 1, ny = B.hi[1] - B.lo[1] + 1;
                for (; i < mine[l].size() && J.parent[l][mine[l][i]] == pb; ++i) {      // chunk ids ascend with their parent's
                    const pltio::BoxI& Cb = meta.levels[l].boxes[mine[l][i]];
                    const int cx = Cb.hi[0] - Cb.lo[0] + 1;
                    for (int k = Cb.lo[2]; k <= Cb.hi[2]; ++k)
                        for (int j = Cb.lo[1]; j <= Cb.hi[1]; ++j) {
                            std::memcpy(dst, tmp.data() + ((long long)(k - B.lo[2]) * ny + (j - B.lo[1])) * nx + (Cb.lo[0] - B.lo[0]), (size_t)cx * 8);
                            dst += cx;
                        }
                }
            }
            check(pa_field_upload_level(fin, l, v, buf[l].comp(v)), "upload");
        }
    }
    check(pa_sync(), "pa_sync");
    M.bar.wait();
    if (talk) std::cout << "Done!" << std::endl;

    if (talk) std::cout << "FillPatching data..." << std::endl;
    for (int l = 0; l < Nlev; ++l) {
        if (talk) std::cout << "on level " << l << std::endl;
        exchange_fill_patch(r, M, fin, ncomp, l, J.ngrow[l], J.interp_type);
        check(pa_fill_patch(fin, 0, ncomp, l, J.ngrow[l], J.interp_type), "pa_fill_patch");
    }
    if (talk) std::cout << "Done!" << std::endl;
    if (talk) std::cout << "Filtering data..." << std::endl;
    for (int l = 0; l < Nlev; ++l) {
        if (talk) std::cout << "on level " << l << std::endl;
        check(pa_filter(fin, 0, fout, 0, ncomp, l, J.filter_type, J.fgr[l]), "pa_filter");
    }
    for (int l = 0; l < Nlev; ++l)
        if (!mine[l].empty())
            for (int c = 0; c < ncomp; ++c) check(pa_field_download_level(fout, l, c, buf[l].comp(c)), "download");
    check(pa_sync(), "pa_sync");
    M.bar.wait();
    if (talk) std::cout << "Done!" << std::endl;

    if (talk) std::cout << "Saving filtered data..." << std::endl;
    char fn[32];
    std::snprintf(fn, sizeof fn, "Cell_D_%05d", r);
    std::vector<pltio::FabRecord> recs;
    for (int l = 0; l < Nlev; ++l) {
        std::vector<const double*> data;
        for (int c = 0; c < ncomp; ++c) data.push_back(buf[l].comp(c));
        auto w = pltio::write_fab_file(J.outfile, meta, l, fn, mine[l], data);
        recs.insert(recs.end(), w.begin(), w.end());
    }
    {
        std::lock_guard<std::mutex> lk(M.mu);
        M.records.insert(M.records.end(), recs.begin(), recs.end());
    }
    pa_field_free(fin); pa_field_free(fout); pa_hier_destroy(h);
    M.bar.wait();
}

// returns after the output plotfile is complete
inline void run_filter_multi(int ngpus, FilterJob& J) {
    J.owner = sfc_owners(*J.meta, J.Nlev, ngpus);
    try { pltio::create_plotfile_dirs(J.outfile, J.Nlev); } catch (std::exception& e) { pa_abort(e.what()); }
    MultiShared M(ngpus);
    std::vector<std::thread> th;
    for (int r = 0; r < ngpus; ++r) th.emplace_back([&, r] {
        try { filter_rank(r, M, J); } catch (std::exception& e) { pa_abort(e.what()); }
    });
    for (auto& t : th) t.join();
    std::vector<int> rr(std::max(J.Nlev - 1, 0), 2);              // write_plotfile hard-codes ref_ratio 2 (filterPlt.cpp:50)
    try { pltio::write_metadata(J.outfile, *J.meta, J.names, J.Nlev, M.records, rr); } catch (std::exception& e) { pa_abort(e.what()); }
    std::cout << "Done!" << std::endl;
}
