// filterPlt3d.b200.ex -- drop-in for PeleAnalysis' filterPlt tool (R/Src/filterPlt.cpp): same ParmParse keys, same plotfile
// in, same output plotfile (<basename(infile)>_filtered in the working directory, grids re-chopped to max_grid_size).  The
// compute block (filterPlt.cpp:166-221: FillPatch ghost cells + Filter::apply_filter) is the C ABI of libpelestencil_b200.
//
//   filterPlt3d.b200.ex infile=<plotfile> [variables=a b c] [max_filter_level=N] [filter_type=1] [base_fgr=2]
//                       [same_fgr_all_levels=0] [max_grid_size=32] [interp_type=1]
//                       [ngpus=N]  (one host thread per GPU, multi_gpu.hpp: the output boxes spread over the GPUs, the
//                                   FillPatch sources of other GPUs moved as packed slabs, one Cell_D file per GPU)
//                       [infiles=a b c]  (a series of plotfiles in one run, series.hpp; every other key applies to each file)
#include <chrono>
#include <cstring>

#include "multi_gpu.hpp"
#include "series.hpp"

static void print_usage(char** argv) {
    std::cerr << "Utility to filter the fields of a pltfile\nusage:\n" << argv[0] << " infile=<s> [options] \n\tOptions:\n"
              << "\t     infile=<s> where s is a pltfile \n"
              << "\t     variables=<s1 s2 s3> variable names to filter [DEF-> all]\n"
              << "\t     max_filter_level=<int> max refinement level to filter, zero-indexed [DEF->1000]\n"
              << "\t     filter_type=<int> filter type as defined in PeleC (1->box, 2->Gaussian, etc) [DEF->1]\n"
              << "\t     base_fgr=<int> filter to grid ratio on the base level, must be even [DEF->2]\n"
              << "\t     same_fgr_all_levels=<bool> keep the same filter to grid ratio on all levels (rather than absolute filter width) [DEF->false]\n"
              << "\t     max_grid_size=<int> AMReX max_grid_size for the output [DEF->32]\n"
              << "\t     interp_type=<int> interpolation when FillPatching: 0 -> piecewise constant, 1 -> cell cons linear [DEF->1]\n";
    std::exit(1);
}

struct FilterKeys {                                    // the keys every file of a run shares
    int finestLevel = 1000, filter_type = 1, base_fgr = 2, max_grid_size = 32, interp_type = 1;
    bool same_fgr = false;
    std::vector<std::string> variables;                // empty: all
};

struct FilterFile {                                    // one plotfile, checked, with its output grids
    std::string infile, outfile;
    pltio::Header H;                                   // the plotfile
    pltio::Header meta;                                // its grids re-chopped to max_grid_size (the output's boxes)
    std::vector<std::vector<int>> parent;              // [level][chunk] -> original box (ascending)
    int Nlev = 0, ngmax = 0;
    std::vector<int> fgr, ngrow;
    std::vector<std::string> names;
};

// the checks of a single run on one plotfile; `who` prefixes every abort message (a series names the file)
static FilterFile filter_file(const FilterKeys& k, const std::string& infile, const std::string& who) {
    FilterFile F;
    F.infile = infile;
    F.outfile = file_root(infile) + "_filtered";
    const pltio::Header& H = F.H;
    try { F.H = pltio::read_header(infile); } catch (std::exception& e) { pa_abort(who + std::string("cannot read plotfile: ") + e.what()); }
    const int Nlev = F.Nlev = std::min(k.finestLevel + 1, H.finest_level + 1);
    if (!k.variables.empty()) {
        F.names = k.variables;
        for (auto& n : F.names)
            if (H.comp(n) < 0) pa_abort(who + "Variable '" + n + "' not found in file");
    } else {
        F.names = H.names;
    }
    // filter-to-grid ratio and ghost width of every level (filterPlt.cpp:138-148), grids re-chopped to max_grid_size (:153)
    F.fgr.resize(Nlev); F.ngrow.resize(Nlev);
    F.meta = H;
    F.parent.resize(Nlev);
    int fgr_lev = k.base_fgr;
    for (int l = 0; l < Nlev; ++l) {
        if (!k.same_fgr && l > 0) {
            const int r = (H.levels[l].domain.hi[0] - H.levels[l].domain.lo[0] + 1) / (H.levels[l - 1].domain.hi[0] - H.levels[l - 1].domain.lo[0] + 1);
            fgr_lev *= r;                                                       // plt_file_data[0]->getRefRatio(lev - 1)
        }
        F.fgr[l] = fgr_lev;
        const int nw = pa_filter_weights(k.filter_type, F.fgr[l], &F.ngrow[l], nullptr, 0);
        if (nw < 0) pa_abort(who + std::string("filter weights: ") + pa_last_error());
        F.ngmax = std::max(F.ngmax, F.ngrow[l]);
        F.meta.levels[l].boxes.clear();
        for (size_t b = 0; b < H.levels[l].boxes.size(); ++b) {
            const pltio::BoxI& B = H.levels[l].boxes[b];
            int one[6] = {B.lo[0], B.lo[1], B.lo[2], B.hi[0], B.hi[1], B.hi[2]};
            const int n = pa_boxes_max_size(1, one, k.max_grid_size, nullptr, 0);
            if (n < 0) pa_abort(who + std::string("max_grid_size: ") + pa_last_error());
            std::vector<int> out(6 * (size_t)n);
            pa_boxes_max_size(1, one, k.max_grid_size, out.data(), n);
            for (int c = 0; c < n; ++c) {
                pltio::BoxI C;
                for (int d = 0; d < 3; ++d) { C.lo[d] = out[6 * c + d]; C.hi[d] = out[6 * c + 3 + d]; }
                F.meta.levels[l].boxes.push_back(C);
                F.parent[l].push_back((int)b);
            }
        }
    }
    return F;
}

// disk -> in[l], every variable on the rank's output boxes, cut from the plotfile boxes they lie in (only those are read)
static void filter_read(const FilterFile& F, const RankCtx& R, HostSet& in, bool talk) {
    const pltio::Header& H = F.H;
    const int ncomp = (int)F.names.size();
    ensure_levels(in, F.Nlev);
    if (talk) std::cout << "Reading data..." << std::endl;
    std::vector<double> tmp;
    for (int l = 0; l < F.Nlev; ++l) {
        if (talk) std::cout << "on level " << l << std::endl;
        const std::vector<int>& mine = R.mine[l];
        std::vector<int> parents;                      // chunk ids ascend with their parent's
        long long np = 0;
        for (int c : mine)
            if (parents.empty() || parents.back() != F.parent[l][c]) {
                parents.push_back(F.parent[l][c]);
                np += H.levels[l].boxes[parents.back()].npts();
            }
        in[l].alloc(R.cells(F.meta, l), ncomp);
        tmp.resize((size_t)np);
        for (int v = 0; v < ncomp; ++v) {
            pltio::read_boxes_comp(F.infile, H, l, H.comp(F.names[v]), parents, tmp.data());
            // each plotfile box becomes the rank's chunks of it, in place
            const double* src = tmp.data();
            double* dst = in[l].comp(v);
            size_t i = 0;
            for (int pb : parents) {
                const pltio::BoxI& B = H.levels[l].boxes[pb];
                const long long nx = B.hi[0] - B.lo[0] + 1, ny = B.hi[1] - B.lo[1] + 1;
                for (; i < mine.size() && F.parent[l][mine[i]] == pb; ++i) {
                    const pltio::BoxI& C = F.meta.levels[l].boxes[mine[i]];
                    const int cx = C.hi[0] - C.lo[0] + 1;
                    for (int kk = C.lo[2]; kk <= C.hi[2]; ++kk)
                        for (int j = C.lo[1]; j <= C.hi[1]; ++j) {
                            std::memcpy(dst, src + ((long long)(kk - B.lo[2]) * ny + (j - B.lo[1])) * nx + (C.lo[0] - B.lo[0]), (size_t)cx * 8);
                            dst += cx;
                        }
                }
                src += B.npts();
            }
        }
    }
}

static void filter_gpu(const FilterKeys& k, const FilterFile& F, const RankCtx& R, HostSet& in, HostSet& out, StagedDownloader& dl, bool talk) {
    const int Nlev = F.Nlev, ncomp = (int)F.names.size();
    const int no_per[3] = {0, 0, 0}, bck[3] = {PA_BC_NEUMANN, PA_BC_NEUMANN, PA_BC_NEUMANN};   // PltFileManager.cpp:118-120: never periodic
    pa_hier* h = R.hier(F.meta, Nlev, no_per, bck, PA_HIER_FILTER_ONLY);
    pa_field *fin = nullptr, *fout = nullptr;
    check(pa_field_alloc(h, ncomp, F.ngmax, &fin), "pa_field_alloc");
    check(pa_field_alloc(h, ncomp, 0, &fout), "pa_field_alloc");
    for (int l = 0; l < Nlev; ++l)
        for (int v = 0; v < ncomp; ++v) check(pa_field_upload_level(fin, l, v, in[l].comp(v)), "upload");
    check(pa_sync(), "pa_sync");
    R.barrier();
    if (talk) std::cout << "Done!" << std::endl;

    if (talk) std::cout << "FillPatching data..." << std::endl;
    for (int l = 0; l < Nlev; ++l) {
        if (talk) std::cout << "on level " << l << std::endl;
        R.fill_patch_exchange(fin, ncomp, l, F.ngrow[l], k.interp_type);
        check(pa_fill_patch(fin, 0, ncomp, l, F.ngrow[l], k.interp_type), "pa_fill_patch");
    }
    if (talk) std::cout << "Done!" << std::endl;
    if (talk) std::cout << "Filtering data..." << std::endl;
    for (int l = 0; l < Nlev; ++l) {
        if (talk) std::cout << "on level " << l << std::endl;
        check(pa_filter(fin, 0, fout, 0, ncomp, l, k.filter_type, F.fgr[l]), "pa_filter");
    }
    ensure_levels(out, Nlev);
    long long mx = 0;
    for (int l = 0; l < Nlev; ++l) {
        if (&out != &in) out[l].alloc(in[l].ncells, ncomp);
        mx = std::max(mx, out[l].ncells);
    }
    dl.reserve(mx);
    for (int l = 0; l < Nlev; ++l)
        for (int c = 0; c < ncomp; ++c) dl.download(fout, l, c, out[l].comp(c), out[l].ncells);
    dl.flush();
    check(pa_sync(), "pa_sync");
    R.barrier();                                       // nobody frees a send slab a peer may still be reading
    if (talk) std::cout << "Done!" << std::endl;
    if (talk) std::cout << "Saving filtered data..." << std::endl;      // the plotfile write follows
    pa_field_free(fin); pa_field_free(fout); pa_hier_destroy(h);
}

int main(int argc, char** argv) {
    if (argc < 2) print_usage(argv);
    ParmParse pp(argc, argv);
    if (pp.contains("help")) print_usage(argv);
    FilterKeys k;
    std::string infile;
    int verbose = 0;
    const bool series = pp.contains("infiles");
    std::vector<std::string> infiles;
    if (series) infiles = series_inputs(pp);
    else pp.get("infile", infile);
    pp.query("max_filter_level", k.finestLevel);
    pp.query("filter_type", k.filter_type);
    pp.query("base_fgr", k.base_fgr);
    pp.query("same_fgr_all_levels", k.same_fgr);
    pp.query("max_grid_size", k.max_grid_size);
    pp.query("interp_type", k.interp_type);
    pp.query("verbose", verbose);
    int ngpus = 1;
    pp.query("ngpus", ngpus);
    if (ngpus < 1) pa_abort("ngpus must be >= 1");
    k.variables.resize(pp.countval("variables"));
    for (size_t i = 0; i < k.variables.size(); ++i) pp.get("variables", k.variables[i], (int)i);

    // progress lines in a single run and from rank 0 of ngpus=N; a series prints none
    const bool talk = !series;
    ToolBody<FilterFile> body;
    body.read = [&](const FilterFile& F, const RankCtx& R, HostSet& in, bool) { filter_read(F, R, in, talk && R.r == 0); };
    body.gpu = [&](const FilterFile& F, const RankCtx& R, HostSet& in, HostSet& out, StagedDownloader& dl) { filter_gpu(k, F, R, in, out, dl, talk && R.r == 0); };

    if (series) {
        // every header read and checked before anything is computed or written; each file runs on one GPU
        std::vector<FilterFile> files;
        for (auto& f : infiles) files.push_back(filter_file(k, f, f + ": "));
        check_distinct_outputs(files);
        run_series(ngpus, files, body, verbose != 0);
        return 0;
    }

    FilterFile F = filter_file(k, infile, "");
    auto t0 = std::chrono::steady_clock::now();
    check(pa_init(0), "pa_init");
    if (ngpus > 1) {
        run_ranks(ngpus, F, body, false, false);
        std::cout << "Done!" << std::endl;
        return 0;
    }
    const RankCtx R(F.meta, F.Nlev);
    // one buffer set holds the inputs and receives the results
    HostSet buf;
    body.read(F, R, buf, true);
    auto t1 = std::chrono::steady_clock::now();
    {
        StagedDownloader dl(0);
        body.gpu(F, R, buf, buf, dl);
    }
    auto t2 = std::chrono::steady_clock::now();

    R.write(F, buf);
    std::cout << "Done!" << std::endl;
    if (verbose) {
        auto s = [](auto a, auto b) { return std::chrono::duration<double>(b - a).count(); };
        std::cout << "[b200] read " << s(t0, t1) << " s, upload+fill+filter+download " << s(t1, t2) << " s, kernels " << pa_kernel_launches() << "\n";
    }
    return 0;
}
