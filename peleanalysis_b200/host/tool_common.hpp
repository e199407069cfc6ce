// tool_common.hpp -- shared plumbing of the two host shells: plotfile metadata -> pa_level_desc, pinned level
// buffers, upload / download, error handling (errors end the process like amrex::Abort).
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <iostream>
#include <string>
#include <vector>

#include "../../include/pele_stencil_b200.h"
#include "parmparse.hpp"
#include "plotfile.hpp"

inline void pa_abort(const std::string& msg) {
    std::cerr << "amrex::Abort::0::" << msg << " !!!" << std::endl;      // same banner the reference prints
    std::exit(1);
}
inline void check(int rc, const char* what) {
    if (rc != PA_OK) pa_abort(std::string(what) + ": " + pa_last_error());
}
inline std::string file_root(const std::string& infile) {          // getFileRoot (grad.cpp:26-31)
    std::string s = infile;
    while (!s.empty() && s.back() == '/') s.pop_back();
    auto p = s.find_last_of('/');
    return p == std::string::npos ? s : s.substr(p + 1);
}

struct HierInput {
    std::vector<pa_level_desc> lv;
    std::vector<std::vector<int>> boxes;
};
inline void make_level_descs(const pltio::Header& h, int nlev, HierInput& out) {
    out.lv.resize(nlev);
    out.boxes.resize(nlev);
    for (int l = 0; l < nlev; ++l) {
        const auto& L = h.levels[l];
        for (int d = 0; d < 3; ++d) {
            out.lv[l].domain_lo[d] = L.domain.lo[d];
            out.lv[l].domain_hi[d] = L.domain.hi[d];
            // Geometry::CellSize = (prob_hi - prob_lo) / N  (AMReX_Geometry.cpp:520), not the rounded header value
            out.lv[l].dx[d] = (h.prob_hi[d] - h.prob_lo[d]) / (double)(L.domain.hi[d] - L.domain.lo[d] + 1);
        }
        for (auto& b : L.boxes) {
            for (int d = 0; d < 3; ++d) out.boxes[l].push_back(b.lo[d]);
            for (int d = 0; d < 3; ++d) out.boxes[l].push_back(b.hi[d]);
        }
        out.lv[l].nboxes = (int)L.boxes.size();
        out.lv[l].boxes = out.boxes[l].data();
        out.lv[l].owner = nullptr;
    }
}

// host buffer holding [comp][level cells].  Pageable by default: measured on the B200 box (profiles/r02_tool_walltime.txt),
// cudaHostAlloc of the tools' buffers costs 0.4 s per GB and as much again to release at exit -- more than the pinned DMA saves on
// data that crosses PCIe once (2 GB pinned for a 50 M-cell grad run: 0.9 s to pin, against 0.2 s of slower copies).  PA_TOOL_PIN=1
// pins them (worth it when the same buffers are reused many times).  alloc() keeps the memory it already holds when that is
// large enough, so a series of plotfiles reuses one buffer per level and grows it only for a larger file.
struct PinnedLevel {
    double* p = nullptr;
    long long ncells = 0;
    int ncomp = 0;
    bool pinned = false;
    size_t cap = 0;                                    // bytes held
    PinnedLevel() = default;
    PinnedLevel(PinnedLevel&& o) noexcept : p(o.p), ncells(o.ncells), ncomp(o.ncomp), pinned(o.pinned), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    PinnedLevel(const PinnedLevel&) = delete;
    PinnedLevel& operator=(const PinnedLevel&) = delete;
    void alloc(long long cells, int comps) {
        ncells = cells; ncomp = comps;
        const size_t bytes = (size_t)cells * comps * 8;
        if (p && bytes <= cap) return;
        release();
        const char* e = std::getenv("PA_TOOL_PIN");
        pinned = e && e[0] == '1';
        cap = bytes;
        if (pinned) {
            void* q = nullptr;
            check(pa_host_alloc(&q, bytes ? bytes : 8), "pa_host_alloc");   // a rank may own no box of a level
            p = (double*)q;
        } else {
            void* q = nullptr;
            if (posix_memalign(&q, 4096, bytes ? bytes : 8) != 0) pa_abort("out of host memory");
            p = (double*)q;
        }
    }
    double* comp(int c) { return p + (long long)c * ncells; }
    const double* comp(int c) const { return p + (long long)c * ncells; }
    void release() { if (p) { if (pinned) pa_host_free(p); else std::free(p); } p = nullptr; cap = 0; }
    ~PinnedLevel() { release(); }
};

using HostSet = std::vector<PinnedLevel>;              // [level] -> [comp][level cells]

inline void ensure_levels(HostSet& s, int nlev) {       // never shrinks: the buffers of deeper levels stay for later files
    if ((int)s.size() < nlev) s.resize(nlev);
}

// Device -> pageable host memory through a pair of pinned bounce buffers: the DMA runs at full PCIe speed into pinned memory and
// the host-side copy of one (level, component) overlaps the transfer of the next.  Measured on the B200 box: a direct download
// into pageable memory ran at 2.2 GB/s (1.6 GB in 0.74 s, profiles/r02_tool_walltime.txt); pinning the whole output instead
// costs 0.4 s per GB to pin and as much to release.  The two buffers hold one component of the largest level each.
class StagedDownloader {
public:
    explicit StagedDownloader(long long max_cells) { reserve(max_cells); }
    ~StagedDownloader() { flush(); free_buffers(); }
    // bounce buffers for levels of up to max_cells cells: kept when they are large enough (a series reuses one downloader)
    void reserve(long long max_cells) {
        if (b_[0] && max_cells <= cap_) return;
        flush();
        free_buffers();
        cap_ = max_cells;
        for (int i = 0; i < 2; ++i) {
            void* q = nullptr;
            check(pa_host_alloc(&q, (size_t)std::max<long long>(cap_, 1) * 8), "pa_host_alloc");
            b_[i] = (double*)q;
        }
    }
    StagedDownloader(const StagedDownloader&) = delete;
    StagedDownloader& operator=(const StagedDownloader&) = delete;
    // queue: component `comp` of level `lev` of `f` -> dst (ncells doubles, pageable or pinned)
    void download(const pa_field* f, int lev, int comp, double* dst, long long ncells) {
        if (ncells > cap_) pa_abort("StagedDownloader: level larger than the bounce buffer");
        const int cur = n_ & 1;
        check(pa_field_download_level(f, lev, comp, b_[cur]), "download");      // asynchronous on the library stream
        if (pend_dst_) copy_out();                                              // host copy of the previous one overlaps this DMA
        check(pa_sync(), "pa_sync");
        pend_dst_ = dst; pend_src_ = b_[cur]; pend_n_ = ncells;
        ++n_;
    }
    void flush() { if (pend_dst_) copy_out(); }
private:
    void free_buffers() { for (int i = 0; i < 2; ++i) if (b_[i]) { pa_host_free(b_[i]); b_[i] = nullptr; } }
    void copy_out() { std::memcpy(pend_dst_, pend_src_, (size_t)pend_n_ * 8); pend_dst_ = nullptr; }
    long long cap_ = 0;
    double* b_[2] = {nullptr, nullptr};
    double* pend_dst_ = nullptr;
    const double* pend_src_ = nullptr;
    long long pend_n_ = 0;
    int n_ = 0;
};
