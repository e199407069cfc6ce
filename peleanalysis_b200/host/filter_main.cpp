// filterPlt3d.b200.ex -- drop-in for PeleAnalysis' filterPlt tool (R/Src/filterPlt.cpp): same ParmParse keys, same plotfile
// in, same output plotfile (<basename(infile)>_filtered in the working directory, grids re-chopped to max_grid_size).  The
// compute block (filterPlt.cpp:166-221: FillPatch ghost cells + Filter::apply_filter) is the C ABI of libpelestencil_b200.
//
//   filterPlt3d.b200.ex infile=<plotfile> [variables=a b c] [max_filter_level=N] [filter_type=1] [base_fgr=2]
//                       [same_fgr_all_levels=0] [max_grid_size=32] [interp_type=1]
//                       [ngpus=N]  (one host thread per GPU, multi_gpu.hpp: the output boxes spread over the GPUs, the
//                                   FillPatch sources of other GPUs moved as packed slabs, one Cell_D file per GPU)
#include <chrono>
#include <cstring>

#include "multi_gpu.hpp"

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

int main(int argc, char** argv) {
    if (argc < 2) print_usage(argv);
    ParmParse pp(argc, argv);
    if (pp.contains("help")) print_usage(argv);
    std::string infile;
    int finestLevel = 1000, filter_type = 1, base_fgr = 2, max_grid_size = 32, interp_type = 1, verbose = 0;
    bool same_fgr = false;
    pp.get("infile", infile);
    pp.query("max_filter_level", finestLevel);
    pp.query("filter_type", filter_type);
    pp.query("base_fgr", base_fgr);
    pp.query("same_fgr_all_levels", same_fgr);
    pp.query("max_grid_size", max_grid_size);
    pp.query("interp_type", interp_type);
    pp.query("verbose", verbose);
    int ngpus = 1;
    pp.query("ngpus", ngpus);
    if (ngpus < 1) pa_abort("ngpus must be >= 1");

    pltio::Header H;
    try { H = pltio::read_header(infile); } catch (std::exception& e) { pa_abort(std::string("cannot read plotfile: ") + e.what()); }
    const int Nlev = std::min(finestLevel + 1, H.finest_level + 1);

    std::vector<std::string> names;
    const int nvar = pp.countval("variables");
    if (nvar > 0) {
        names.resize(nvar);
        for (int i = 0; i < nvar; ++i) {
            pp.get("variables", names[i], i);
            if (H.comp(names[i]) < 0) pa_abort("Variable '" + names[i] + "' not found in file");
        }
    } else {
        names = H.names;
    }
    const int ncomp = (int)names.size();

    auto t0 = std::chrono::steady_clock::now();
    check(pa_init(0), "pa_init");
    // filter-to-grid ratio and ghost width of every level (filterPlt.cpp:138-148), grids re-chopped to max_grid_size (:153)
    std::vector<int> fgr(Nlev), ngrow(Nlev);
    pltio::Header meta = H;
    std::vector<std::vector<std::vector<pltio::BoxI>>> chunks(Nlev);           // [level][original box] -> its chunks
    std::vector<std::vector<int>> parent(Nlev);                                 // [level][chunk] -> original box
    int fgr_lev = base_fgr, ngmax = 0;
    for (int l = 0; l < Nlev; ++l) {
        if (!same_fgr && l > 0) {
            const int r = (H.levels[l].domain.hi[0] - H.levels[l].domain.lo[0] + 1) / (H.levels[l - 1].domain.hi[0] - H.levels[l - 1].domain.lo[0] + 1);
            fgr_lev *= r;                                                       // plt_file_data[0]->getRefRatio(lev - 1)
        }
        fgr[l] = fgr_lev;
        const int nw = pa_filter_weights(filter_type, fgr[l], &ngrow[l], nullptr, 0);
        if (nw < 0) pa_abort(std::string("filter weights: ") + pa_last_error());
        ngmax = std::max(ngmax, ngrow[l]);
        meta.levels[l].boxes.clear();
        chunks[l].resize(H.levels[l].boxes.size());
        for (size_t b = 0; b < H.levels[l].boxes.size(); ++b) {
            const pltio::BoxI& B = H.levels[l].boxes[b];
            int one[6] = {B.lo[0], B.lo[1], B.lo[2], B.hi[0], B.hi[1], B.hi[2]};
            const int n = pa_boxes_max_size(1, one, max_grid_size, nullptr, 0);
            if (n < 0) pa_abort(std::string("max_grid_size: ") + pa_last_error());
            std::vector<int> out(6 * (size_t)n);
            pa_boxes_max_size(1, one, max_grid_size, out.data(), n);
            for (int c = 0; c < n; ++c) {
                pltio::BoxI C;
                for (int d = 0; d < 3; ++d) { C.lo[d] = out[6 * c + d]; C.hi[d] = out[6 * c + 3 + d]; }
                chunks[l][b].push_back(C);
                meta.levels[l].boxes.push_back(C);
                parent[l].push_back((int)b);
            }
        }
    }
    const std::string outfile = file_root(infile) + "_filtered";
    if (ngpus > 1) {
        FilterJob J;
        J.infile = infile; J.outfile = outfile; J.H = &H; J.meta = &meta; J.parent = parent; J.Nlev = Nlev;
        J.filter_type = filter_type; J.interp_type = interp_type; J.ngmax = ngmax; J.fgr = fgr; J.ngrow = ngrow; J.names = names;
        run_filter_multi(ngpus, J);
        return 0;
    }
    HierInput hi;
    make_level_descs(meta, Nlev, hi);
    const int no_per[3] = {0, 0, 0}, bck[3] = {PA_BC_NEUMANN, PA_BC_NEUMANN, PA_BC_NEUMANN};   // PltFileManager.cpp:118-120: never periodic
    pa_hier* h = nullptr;
    check(pa_hier_create2(&h, Nlev, hi.lv.data(), no_per, bck, 0, 1, PA_HIER_FILTER_ONLY), "pa_hier_create");
    pa_field *fin = nullptr, *fout = nullptr;
    check(pa_field_alloc(h, ncomp, ngmax, &fin), "pa_field_alloc");
    check(pa_field_alloc(h, ncomp, 0, &fout), "pa_field_alloc");

    std::cout << "Reading data..." << std::endl;
    std::vector<PinnedLevel> buf(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        std::cout << "on level " << l << std::endl;
        const long long nc = H.levels[l].ncells();
        buf[l].alloc(nc, ncomp);
        std::vector<double> tmp((size_t)nc);
        for (int v = 0; v < ncomp; ++v) {
            pltio::read_level_comp(infile, H, l, H.comp(names[v]), tmp.data());
            // the plotfile's FABs cut into the output boxes: each original box becomes its chunks, in place
            const double* src = tmp.data();
            double* dst = buf[l].comp(v);
            for (size_t b = 0; b < H.levels[l].boxes.size(); ++b) {
                const pltio::BoxI& B = H.levels[l].boxes[b];
                const long long nx = B.hi[0] - B.lo[0] + 1, ny = B.hi[1] - B.lo[1] + 1;
                for (const pltio::BoxI& C : chunks[l][b]) {
                    const int cx = C.hi[0] - C.lo[0] + 1;
                    for (int k = C.lo[2]; k <= C.hi[2]; ++k)
                        for (int j = C.lo[1]; j <= C.hi[1]; ++j) {
                            std::memcpy(dst, src + ((long long)(k - B.lo[2]) * ny + (j - B.lo[1])) * nx + (C.lo[0] - B.lo[0]), (size_t)cx * 8);
                            dst += cx;
                        }
                }
                src += B.npts();
            }
            check(pa_field_upload_level(fin, l, v, buf[l].comp(v)), "upload");
        }
    }
    check(pa_sync(), "pa_sync");
    std::cout << "Done!" << std::endl;
    auto t1 = std::chrono::steady_clock::now();

    std::cout << "FillPatching data..." << std::endl;
    for (int l = 0; l < Nlev; ++l) {
        std::cout << "on level " << l << std::endl;
        check(pa_fill_patch(fin, 0, ncomp, l, ngrow[l], interp_type), "pa_fill_patch");
    }
    std::cout << "Done!" << std::endl;
    std::cout << "Filtering data..." << std::endl;
    for (int l = 0; l < Nlev; ++l) {
        std::cout << "on level " << l << std::endl;
        check(pa_filter(fin, 0, fout, 0, ncomp, l, filter_type, fgr[l]), "pa_filter");
    }
    {
        long long mx = 0;
        for (int l = 0; l < Nlev; ++l) mx = std::max(mx, buf[l].ncells);
        StagedDownloader dl(mx);
        for (int l = 0; l < Nlev; ++l)
            for (int c = 0; c < ncomp; ++c) dl.download(fout, l, c, buf[l].comp(c), buf[l].ncells);
        dl.flush();
    }
    check(pa_sync(), "pa_sync");
    std::cout << "Done!" << std::endl;
    auto t2 = std::chrono::steady_clock::now();

    std::cout << "Saving filtered data..." << std::endl;
    std::vector<std::vector<const double*>> data(Nlev);
    for (int l = 0; l < Nlev; ++l) for (int c = 0; c < ncomp; ++c) data[l].push_back(buf[l].comp(c));
    std::vector<int> rr(std::max(Nlev - 1, 0), 2);            // write_plotfile hard-codes ref_ratio 2 (filterPlt.cpp:50)
    try { pltio::write_plotfile(outfile, meta, names, data, rr); } catch (std::exception& e) { pa_abort(e.what()); }
    std::cout << "Done!" << std::endl;
    if (verbose) {
        auto s = [](auto a, auto b) { return std::chrono::duration<double>(b - a).count(); };
        std::cout << "[b200] read+upload " << s(t0, t1) << " s, fill+filter+download " << s(t1, t2) << " s, kernels " << pa_kernel_launches() << "\n";
    }
    pa_field_free(fin); pa_field_free(fout); pa_hier_destroy(h);
    return 0;
}
