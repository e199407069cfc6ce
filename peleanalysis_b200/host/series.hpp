// series.hpp -- a series of plotfiles in one process (key infiles=plt00100 plt00200 ...): CUDA start-up is paid once, and on
// every GPU the disk read of file k+1 and the plotfile write of file k-1 overlap the GPU work on file k.
//
// Each GPU has one worker of three threads:
//   reader  takes the next file of the list (files are handed out in list order, one shared counter over all workers) and
//           reads it into a free input set of host buffers;
//   GPU     (the worker thread) runs the tool's per-file body on its device: hierarchy and fields created, upload, the
//           library calls, download into a free output set, hierarchy and fields freed;
//   writer  writes the output set as the file's plotfile.
// All three run the body with a one-rank RankCtx (multi_gpu.hpp), as a single run does.
// Host memory: 2 input sets and 2 output sets per worker, each one PinnedLevel per level, allocated on first use and grown
// only when a larger file arrives, so a worker holds at most 4 buffer sets of the largest file.  They stay pageable
// (tool_common.hpp: pinning costs more than it saves on data that crosses PCIe once); the pinned bounce buffers of the
// StagedDownloader are allocated once per worker.  Hierarchies and fields are not cached: building them is a small part of a
// file's time, and each file goes through exactly the calls of a single run, so its output is byte-identical to that run's.
#pragma once
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <map>
#include <mutex>
#include <thread>

#include "multi_gpu.hpp"

// infiles=...: the list.  The keys that name one file cannot be combined with it, and transport only concerns box
// distribution of one file over several GPUs.
inline std::vector<std::string> series_inputs(const ParmParse& pp) {
    std::vector<std::string> in(pp.countval("infiles"));
    for (size_t i = 0; i < in.size(); ++i) pp.get("infiles", in[i], (int)i);
    if (in.empty()) pa_abort("infiles needs at least one plotfile");
    for (const char* k : {"infile", "outfile", "transport"})
        if (pp.contains(k)) pa_abort(std::string("infiles cannot be combined with ") + k + " (each file's output has its default name)");
    return in;
}

// before anything is computed: every output name once (two inputs of the same root name would overwrite each other)
template <class File>
void check_distinct_outputs(const std::vector<File>& files) {
    std::map<std::string, std::string> seen;
    for (const File& F : files) {
        auto r = seen.emplace(F.outfile, F.infile);
        if (!r.second) pa_abort("infiles: " + r.first->second + " and " + F.infile + " both write " + F.outfile);
    }
}

template <class T>
class Channel {
public:
    void push(T v) {
        { std::lock_guard<std::mutex> lk(mu_); q_.push_back(std::move(v)); }
        cv_.notify_one();
    }
    T pop() {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return !q_.empty(); });
        T v = std::move(q_.front());
        q_.pop_front();
        return v;
    }
private:
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<T> q_;
};

struct SeriesShared {
    std::atomic<int> next{0};                          // next file of the list to hand out
    std::mutex print;
};

template <class File>
void series_worker(int dev, SeriesShared& S, const std::vector<File>& files, const ToolBody<File>& body, bool verbose) {
    struct Item { int file, set; double read_s, gpu_s; int64_t dev_bytes; };
    using clk = std::chrono::steady_clock;
    auto since = [](clk::time_point t) { return std::chrono::duration<double>(clk::now() - t).count(); };
    auto stage = [&](const File& F, const std::function<void()>& fn) {
        try { fn(); } catch (std::exception& e) { pa_abort(F.infile + ": " + e.what()); }
    };
    check(pa_init(dev), "pa_init");
    HostSet in[2], out[2];
    Channel<int> free_in, free_out;
    Channel<Item> to_gpu, to_write;
    for (int i = 0; i < 2; ++i) { free_in.push(i); free_out.push(i); }

    std::thread reader([&] {
        for (;;) {
            const int k = S.next++;
            if (k >= (int)files.size()) { to_gpu.push(Item{-1, -1, 0, 0, 0}); return; }
            const int s = free_in.pop();
            const auto t0 = clk::now();
            stage(files[k], [&] { body.read(files[k], RankCtx(files[k].meta, files[k].Nlev), in[s], false); });
            to_gpu.push(Item{k, s, since(t0), 0, 0});
        }
    });
    std::thread writer([&] {
        for (;;) {
            const Item it = to_write.pop();
            if (it.file < 0) return;
            const File& F = files[it.file];
            const auto t0 = clk::now();
            stage(F, [&] { RankCtx(F.meta, F.Nlev).write(F, out[it.set]); });
            const double write_s = since(t0);
            free_out.push(it.set);
            if (verbose) {
                std::lock_guard<std::mutex> lk(S.print);
                std::cout << "[b200] series " << it.file + 1 << "/" << files.size() << " " << F.infile << " -> " << F.outfile << " on GPU " << dev
                          << ": read " << it.read_s << " s, gpu " << it.gpu_s << " s, write " << write_s << " s, device bytes " << it.dev_bytes
                          << std::endl;
            }
        }
    });
    StagedDownloader dl(0);
    for (;;) {
        Item it = to_gpu.pop();
        if (it.file < 0) { to_write.push(it); break; }
        const int o = free_out.pop();
        const auto t0 = clk::now();
        const File& F = files[it.file];
        stage(F, [&] { body.gpu(F, RankCtx(F.meta, F.Nlev), in[it.set], out[o], dl); });
        it.gpu_s = since(t0);
        free_in.push(it.set);
        check(pa_debug_device_bytes(&it.dev_bytes), "pa_debug_device_bytes");
        it.set = o;
        to_write.push(it);
    }
    reader.join();
    writer.join();
}

// returns after every output plotfile is complete; ngpus workers (one per GPU) share the list
template <class File>
void run_series(int ngpus, const std::vector<File>& files, const ToolBody<File>& body, bool verbose) {
    if (ngpus < 1) pa_abort("ngpus must be >= 1");
    SeriesShared S;
    const int nw = std::min<int>(ngpus, (int)files.size());
    std::vector<std::thread> th;
    for (int r = 0; r < nw; ++r) th.emplace_back([&, r] { series_worker(r, S, files, body, verbose); });
    for (auto& t : th) t.join();
}
