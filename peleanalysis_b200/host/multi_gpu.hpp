// multi_gpu.hpp -- the grad, curvature and filterPlt tools on several GPUs of one node from ONE process: one host thread per
// GPU, no MPI, no NCCL.
//
// What an MPI build of the reference does rank by rank (boxes distributed by DistributionMapping, ghost cells through
// FillBoundary / ParallelCopy, one Cell_D file per rank) is done here thread by thread.  Each thread runs the tool's per-file
// read, GPU and write functions -- the same ones a single run and every file of a series run -- with a RankCtx of its own:
// thread r owns GPU r and the boxes the SFC distribution gives rank r, reads only those from disk, moves the ghost sources
// owned by other threads as packed slabs with device-to-device copies (pa_copy_async), runs the tool's C-ABI calls, and
// writes its own boxes to Level_l/Cell_D_<r>; Header and Cell_H are written once every thread is done.  Barriers between
// threads stand where the reference has MPI synchronisation: before anyone reads a peer's slab, and before anyone frees a
// slab a peer may still read.  At one rank none of these cross-rank steps makes a library call.
// grad and curvature have two transports (key transport=peer|slab): with peer links (the default) every thread also maps the
// other threads' level slabs (pa_field_map_peer_ptr) and the stencil kernels read cross-GPU neighbour faces and coarse cells in
// place over NVLink, so only the ragged remainder travels in the slabs; with transport=slab no field slab is mapped and every
// ghost source of another thread travels in the slabs (the width-1 exchange plan of hier.cpp: build_exchange), as filterPlt's
// FillPatch sources always do.  Every transport enables peer access between the GPUs: it lets the copy engines move the
// pa_copy_async copies GPU to GPU directly instead of through host memory.
#pragma once
#include <condition_variable>
#include <cstdio>
#include <functional>
#include <mutex>
#include <thread>
#include <utility>

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
    std::vector<std::vector<const double*>> slab;      // [rank][field * nlev + level]: level slabs, published for the peers
    std::vector<double*> send;                         // [rank]: send slab
    std::vector<std::vector<int64_t>> soff;            // [rank][peer .. ]: offsets into it
    std::vector<pltio::FabRecord> records;             // what every thread wrote
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

// the reference tools hard-code ref_ratio 2 in the plotfiles they write (grad.cpp:255, curvature.cpp:842, filterPlt.cpp:50)
inline std::vector<int> ref_ratio_line(int nlev) { return std::vector<int>(std::max(nlev - 1, 0), 2); }

// The rank a tool's per-file functions run as, and the cross-rank steps they take.  The cross-rank steps are collective: every
// rank calls them in the same order.  At n == 1 (a single run, every file of a series) the rank owns every box and write() is
// the only step that does anything, so the one-GPU launch sequence has no exchange in it.
// A tool's File has infile, outfile, Nlev, names (the output's components) and meta (the output's grids and header).
struct RankCtx {
    int r = 0, n = 1;
    bool peer_links = false;                           // n > 1 and transport=peer: peer slabs are mapped and read in place
    MultiShared* M = nullptr;                          // shared by the n threads; null when n == 1
    std::vector<std::vector<int>> owner;               // [level][box] -> rank
    std::vector<std::vector<int>> mine;                // [level] -> the boxes this rank owns, ascending

    RankCtx(int r, int n, std::vector<std::vector<int>> owner_, MultiShared* M, bool peer)
        : r(r), n(n), peer_links(n > 1 && peer), M(M), owner(std::move(owner_)), mine(owner.size()) {
        for (size_t l = 0; l < owner.size(); ++l)
            for (int b = 0; b < (int)owner[l].size(); ++b)
                if (owner[l][b] == r) mine[l].push_back(b);
    }
    // the one rank of a run on one GPU: every box of `grids`
    RankCtx(const pltio::Header& grids, int nlev) : RankCtx(0, 1, all_on_rank0(grids, nlev), nullptr, false) {}

    long long cells(const pltio::Header& grids, int l) const {          // this rank's cells of level l
        long long nc = 0;
        for (int b : mine[l]) nc += grids.levels[l].boxes[b].npts();
        return nc;
    }

    // this rank's hierarchy over `grids` (PA_HIER_PEER_LINKS added with peer links)
    pa_hier* hier(const pltio::Header& grids, int nlev, const int is_per[3], const int bck[3], unsigned flags) const {
        HierInput hi;
        make_level_descs(grids, nlev, hi);
        for (int l = 0; l < nlev; ++l) hi.lv[l].owner = owner[l].data();
        pa_hier* h = nullptr;
        check(pa_hier_create2(&h, nlev, hi.lv.data(), is_per, bck, r, n, flags | (peer_links ? PA_HIER_PEER_LINKS : 0u)), "pa_hier_create");
        return h;
    }

    // with peer links: every thread publishes the level slabs of its fields, then maps everyone else's (all threads pass the
    // same number of fields in the same order)
    void map_peers(int nlev, const std::vector<pa_field*>& fields) const {
        if (!peer_links) return;
        M->slab[r].assign(fields.size() * nlev, nullptr);
        for (size_t f = 0; f < fields.size(); ++f)
            for (int l = 0; l < nlev; ++l) check(pa_field_slab(fields[f], l, &M->slab[r][f * nlev + l]), "pa_field_slab");
        M->bar.wait();
        for (int p = 0; p < n; ++p)
            if (p != r)
                for (size_t f = 0; f < fields.size(); ++f)
                    for (int l = 0; l < nlev; ++l) {
                        check(pa_field_map_peer_ptr(fields[f], l, p, M->slab[p][f * nlev + l]), "pa_field_map_peer_ptr");
                        ++M->mapped[r];
                    }
        M->bar.wait();
    }

    // The cross-rank step in front of a ghost fill of components comp .. comp+ncomp-1 of f: what the neighbour links do not
    // cover -- ragged same-level neighbours, coarse cells of coarse-fine faces owned by another rank -- moves as packed slabs
    // (the width-1 exchange plan).  Its first barrier is also the ordering point peer links need: every rank has finished
    // (pa_sync) whatever wrote the data its peers are about to read.
    void exchange(pa_field* f, int comp, int ncomp) const {
        if (n == 1) return;
        transfer("exchange",
                 [&](double** s, double** rv, int64_t* so, int64_t* ro) { check(pa_exchange_buffers(f, ncomp, s, rv, so, ro), "pa_exchange_buffers"); },
                 [&] { check(pa_exchange_pack(f, comp, ncomp), "pa_exchange_pack"); },
                 [&] { check(pa_exchange_mark_received(f, comp, ncomp), "pa_exchange_mark_received"); });
    }

    // the same in front of pa_fill_patch(lev): the FillPatch sources of level lev owned by other ranks (the filterPlt
    // hierarchy has no peer links, so nothing is read in place)
    void fill_patch_exchange(pa_field* f, int ncomp, int lev, int nghost, int interp_type) const {
        if (n == 1) return;
        transfer("FillPatch",
                 [&](double** s, double** rv, int64_t* so, int64_t* ro) {
                     check(pa_fill_patch_exchange_buffers(f, ncomp, lev, nghost, interp_type, s, rv, so, ro), "pa_fill_patch_exchange_buffers");
                 },
                 [&] { check(pa_fill_patch_pack(f, 0, ncomp, lev, nghost, interp_type), "pa_fill_patch_pack"); },
                 [&] { check(pa_fill_patch_mark_received(f, 0, ncomp, lev, nghost, interp_type), "pa_fill_patch_mark_received"); });
    }

    void barrier() const { if (M) M->bar.wait(); }

    // this rank's share of F's output plotfile from components 0 .. names-1 of out[l]: at n == 1 the whole plotfile with up
    // to four writer threads per level (pltio::write_plotfile); at n > 1 the rank's boxes into Level_l/Cell_D_<r>, whose
    // records run_ranks turns into Header and Cell_H
    template <class File>
    void write(const File& F, const HostSet& out) const {
        std::vector<std::vector<const double*>> data(F.Nlev);
        for (int l = 0; l < F.Nlev; ++l)
            for (size_t c = 0; c < F.names.size(); ++c) data[l].push_back(out[l].comp((int)c));
        if (n == 1) {
            try { pltio::write_plotfile(F.outfile, F.meta, F.names, data, ref_ratio_line(F.Nlev)); } catch (std::exception& e) { pa_abort(e.what()); }
            return;
        }
        char fn[32];
        std::snprintf(fn, sizeof fn, "Cell_D_%05d", r);
        std::vector<pltio::FabRecord> recs;
        for (int l = 0; l < F.Nlev; ++l) {
            auto w = pltio::write_fab_file(F.outfile, F.meta, l, fn, mine[l], data[l]);
            recs.insert(recs.end(), w.begin(), w.end());
        }
        std::lock_guard<std::mutex> lk(M->mu);
        M->records.insert(M->records.end(), recs.begin(), recs.end());
    }

private:
    static std::vector<std::vector<int>> all_on_rank0(const pltio::Header& grids, int nlev) {
        std::vector<std::vector<int>> o(nlev);
        for (int l = 0; l < nlev; ++l) o[l].assign(grids.levels[l].boxes.size(), 0);
        return o;
    }

    // one exchange plan: buffers -> pack -> device-to-device copies of each peer's segment -> mark
    template <class Buffers, class Pack, class Mark>
    void transfer(const char* plan, Buffers buffers, Pack pack, Mark mark) const {
        double *send = nullptr, *recv = nullptr;
        std::vector<int64_t> so(n + 1), ro(n + 1);
        buffers(&send, &recv, so.data(), ro.data());
        pack();
        check(pa_sync(), "pa_sync");
        M->send[r] = send;
        M->soff[r] = so;
        M->bar.wait();
        for (int p = 0; p < n; ++p) {
            if (p == r) continue;
            const int64_t cnt = ro[p + 1] - ro[p];
            if (cnt != M->soff[p][r + 1] - M->soff[p][r]) pa_abort(std::string("multi-GPU ") + plan + " plan: send / recv counts disagree");
            if (cnt > 0) check(pa_copy_async(recv + ro[p], M->send[p] + M->soff[p][r], cnt), "pa_copy_async");
        }
        M->received[r] += ro[n];
        mark();
        check(pa_sync(), "pa_sync");
        M->bar.wait();                                 // the send slabs may be repacked from here on
    }
};

// A tool's per-file body, run by a single run, by every thread of ngpus=N (run_ranks) and for every file of a series
// (series.hpp).  read() fills `in` with the rank's boxes of the inputs; in_place: `in` receives the results too, so it gets
// their components as well.  gpu() runs on a thread that called pa_init for its device, leaves nothing allocated on the device,
// and fills `out` (which may be `in`).  RankCtx::write writes `out`.
template <class File>
struct ToolBody {
    std::function<void(const File&, const RankCtx&, HostSet& in, bool in_place)> read;
    std::function<void(const File&, const RankCtx&, HostSet& in, HostSet& out, StagedDownloader& dl)> gpu;
};

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

// ngpus=N on one plotfile: thread r runs the body on GPU r as rank r of N.  peer: transport=peer; report: print the transport
// line.  Returns after the output plotfile is complete.
template <class File>
void run_ranks(int ngpus, const File& F, const ToolBody<File>& body, bool peer, bool report) {
    const std::vector<std::vector<int>> owner = sfc_owners(F.meta, F.Nlev, ngpus);
    try { pltio::create_plotfile_dirs(F.outfile, F.Nlev); } catch (std::exception& e) { pa_abort(e.what()); }
    MultiShared M(ngpus);
    std::vector<std::thread> th;
    for (int r = 0; r < ngpus; ++r) th.emplace_back([&, r] {
        try {
            check(pa_init(r), "pa_init");
            for (int p = 0; p < ngpus; ++p) if (p != r) check(pa_enable_peer_access(p), "pa_enable_peer_access");
            const RankCtx R(r, ngpus, owner, &M, peer);
            HostSet buf;                               // holds the inputs and receives the results
            StagedDownloader dl(0);
            body.read(F, R, buf, true);
            body.gpu(F, R, buf, buf, dl);
            R.write(F, buf);
        } catch (std::exception& e) { pa_abort(e.what()); }
    });
    for (auto& t : th) t.join();
    if (report) print_transport_report(M, peer);
    try { pltio::write_metadata(F.outfile, F.meta, F.names, F.Nlev, M.records, ref_ratio_line(F.Nlev)); } catch (std::exception& e) { pa_abort(e.what()); }
}
