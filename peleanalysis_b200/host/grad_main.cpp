// grad3d.b200.ex -- drop-in for PeleAnalysis' grad tool (R/Src/grad.cpp): same ParmParse keys, same plotfile in/out,
// same output variable names; the operator block (grad.cpp:151-236) is the C ABI of libpelestencil_b200.
//
//   grad3d.b200.ex infile=<plotfile> [gradVar=temp] [finestLevel=N] [Aux_Variables=a b ...] [is_per=1 1 1]
//                  [sym_dir=0 0 0] [outfile=<name>]          extensions: gradVars=a b c  (several variables, one pass)
//                                                                        ngpus=N  (one host thread per GPU, multi_gpu.hpp)
//                                                                        transport=peer|slab  (with ngpus=N: peer links +
//                                                                        packed slabs, or packed slabs only)
//                                                                        infiles=a b c  (a series of plotfiles in one run,
//                                                                        series.hpp; every other key applies to each file)
#include <chrono>

#include "multi_gpu.hpp"
#include "series.hpp"

static void print_usage(char** argv) {
    std::cerr << "usage:\n" << argv[0] << " infile=<plotfilename> \n\tOptions:\n\tis_per=<L M N> gradVar=<name>\n";
    std::exit(1);
}

struct GradOpts {                                      // the keys every file of a run shares
    int finestLevel = 1000;
    std::vector<std::string> gvars, aux;
    std::vector<int> is_per;
    int bck[3];
};

struct GradFile {                                      // one plotfile, checked
    std::string infile, outfile;
    pltio::Header H, meta;                             // the plotfile; the output's header (time 0, grad.cpp:256)
    int Nlev = 0;
    std::vector<std::string> names;
    int nv = 0, nIn = 0, nOut = 0;
};

// the checks of a single run on one plotfile; `who` prefixes every abort message (a series names the file)
static GradFile grad_file(const GradOpts& o, const std::string& infile, const std::string& who) {
    GradFile F;
    F.infile = infile;
    try { F.H = pltio::read_header(infile); } catch (std::exception& e) { pa_abort(who + std::string("cannot read plotfile: ") + e.what()); }
    F.Nlev = std::min(o.finestLevel, F.H.finest_level) + 1;
    for (auto& v : o.gvars)
        if (F.H.comp(v) < 0) { std::cout << "Cannot find " << v << " data in pltfile \n"; pa_abort(who + "Cannot find " + v + " data in pltfile"); }
    for (auto& a : o.aux)
        if (F.H.comp(a) < 0) pa_abort(who + "Unknown auxiliary variable name: " + a);
    F.nv = (int)o.gvars.size();
    F.nIn = F.nv + (int)o.aux.size();
    F.nOut = F.nIn + 4 * F.nv;
    for (auto& v : o.gvars) F.names.push_back(v);
    for (auto& a : o.aux) F.names.push_back(a);
    for (auto& v : o.gvars) { F.names.push_back(v + "_gx"); F.names.push_back(v + "_gy"); F.names.push_back(v + "_gz"); F.names.push_back("||grad" + v + "||"); }
    F.outfile = file_root(infile) + "_gt";
    F.meta = F.H;
    F.meta.time = 0.0;                                 // WriteMultiLevelPlotfile(..., 0.0, ...) (grad.cpp:256)
    return F;
}

// disk -> in[l] components 0 .. nIn-1 (gradient variables, then pass-through variables) of the rank's boxes; in_place: room
// for the results as well
static void grad_read(const GradOpts& o, const GradFile& F, const RankCtx& R, HostSet& in, bool in_place, bool talk) {
    ensure_levels(in, F.Nlev);
    for (int l = 0; l < F.Nlev; ++l) {
        if (talk) std::cout << "Reading data for level: " << l << std::endl;
        in[l].alloc(R.cells(F.H, l), in_place ? F.nOut : F.nIn);
        for (int v = 0; v < F.nv; ++v) pltio::read_boxes_comp(F.infile, F.H, l, F.H.comp(o.gvars[v]), R.mine[l], in[l].comp(v));
        for (size_t a = 0; a < o.aux.size(); ++a) pltio::read_boxes_comp(F.infile, F.H, l, F.H.comp(o.aux[a]), R.mine[l], in[l].comp(F.nv + (int)a));
    }
}

// the gradient variables to the device, pa_grad, the results into out[l] components nIn .. nOut-1 (the inputs copied over
// when out is another set)
static void grad_gpu(const GradOpts& o, const GradFile& F, const RankCtx& R, HostSet& in, HostSet& out, StagedDownloader& dl) {
    const int Nlev = F.Nlev, nv = F.nv;
    pa_hier* h = R.hier(F.H, Nlev, o.is_per.data(), o.bck, 0);
    pa_field *fin = nullptr, *fout = nullptr;
    check(pa_field_alloc(h, nv, 1, &fin), "pa_field_alloc");
    check(pa_field_alloc(h, 4 * nv, 0, &fout), "pa_field_alloc");
    for (int l = 0; l < Nlev; ++l)
        for (int v = 0; v < nv; ++v) check(pa_field_upload_level(fin, l, v, in[l].comp(v)), "upload");
    R.map_peers(Nlev, {fin});
    R.exchange(fin, 0, nv);
    check(pa_grad(fin, 0, nv, fout, 0), "pa_grad");
    ensure_levels(out, Nlev);
    long long mx = 0;
    for (int l = 0; l < Nlev; ++l) {
        const long long nc = in[l].ncells;
        mx = std::max(mx, nc);
        if (&out != &in) {
            out[l].alloc(nc, F.nOut);
            std::memcpy(out[l].comp(0), in[l].comp(0), (size_t)F.nIn * nc * 8);
        }
    }
    dl.reserve(mx);
    for (int l = 0; l < Nlev; ++l)
        for (int c = 0; c < 4 * nv; ++c) dl.download(fout, l, c, out[l].comp(F.nIn + c), out[l].ncells);
    dl.flush();
    check(pa_sync(), "pa_sync");
    R.barrier();                                       // nobody frees a slab (or send slab) a peer may still be reading
    pa_field_free(fin); pa_field_free(fout); pa_hier_destroy(h);
}

int main(int argc, char** argv) {
    if (argc < 2) print_usage(argv);
    ParmParse pp(argc, argv);
    if (pp.contains("help")) print_usage(argv);
    GradOpts o;
    std::string infile, gradVar = "temp";
    int verbose = 0;
    const bool series = pp.contains("infiles");
    std::vector<std::string> infiles;
    if (series) infiles = series_inputs(pp);
    else pp.get("infile", infile);
    pp.query("gradVar", gradVar);
    pp.query("finestLevel", o.finestLevel);
    pp.query("verbose", verbose);

    int ng = pp.countval("gradVars");
    if (ng > 0) { o.gvars.resize(ng); for (int i = 0; i < ng; ++i) pp.get("gradVars", o.gvars[i], i); }
    else o.gvars.push_back(gradVar);
    o.aux.resize(pp.countval("Aux_Variables"));
    for (size_t i = 0; i < o.aux.size(); ++i) pp.get("Aux_Variables", o.aux[i], (int)i);
    std::vector<int> sym_dir(3, 0);
    o.is_per.assign(3, 1);
    pp.queryarr("sym_dir", sym_dir, 0, 3);
    pp.queryarr("is_per", o.is_per, 0, 3);
    for (int d = 0; d < 3; ++d) o.bck[d] = sym_dir[d] ? PA_BC_REFLECT_ODD : PA_BC_NEUMANN;
    int ngpus = 1;
    pp.query("ngpus", ngpus);

    // the threads of ngpus=N and the files of a series print no progress lines
    ToolBody<GradFile> body;
    body.read = [&](const GradFile& F, const RankCtx& R, HostSet& in, bool in_place) { grad_read(o, F, R, in, in_place, false); };
    body.gpu = [&](const GradFile& F, const RankCtx& R, HostSet& in, HostSet& out, StagedDownloader& dl) { grad_gpu(o, F, R, in, out, dl); };

    if (series) {
        // every header read and checked before anything is computed or written
        std::vector<GradFile> files;
        for (auto& f : infiles) files.push_back(grad_file(o, f, f + ": "));
        check_distinct_outputs(files);
        std::cout << "Periodicity assumed for this case: ";
        for (int d = 0; d < 3; ++d) std::cout << o.is_per[d] << " ";
        std::cout << "\n";
        run_series(ngpus, files, body, verbose != 0);
        return 0;
    }

    GradFile F = grad_file(o, infile, "");
    std::cout << "Periodicity assumed for this case: ";
    for (int d = 0; d < 3; ++d) std::cout << o.is_per[d] << " ";
    std::cout << "\n";
    pp.query("outfile", F.outfile);

    std::string transport = "peer";
    pp.query("transport", transport);
    if (transport != "peer" && transport != "slab") pa_abort("transport must be peer or slab (got " + transport + ")");
    if (ngpus > 1) {
        std::cout << "Writing new data to " << F.outfile << std::endl;
        run_ranks(ngpus, F, body, transport == "peer", verbose != 0);
        return 0;
    }
    auto tnow = [] { return std::chrono::steady_clock::now(); };
    auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
    auto t0 = tnow();
    check(pa_init(0), "pa_init");
    auto t1 = tnow();
    const RankCtx R(F.meta, F.Nlev);
    // one buffer set holds the inputs and receives the results
    HostSet buf;
    grad_read(o, F, R, buf, true, true);
    auto t2 = tnow();
    {
        StagedDownloader dl(0);
        grad_gpu(o, F, R, buf, buf, dl);
    }
    auto t3 = tnow();
    std::cout << "Writing new data to " << F.outfile << std::endl;
    R.write(F, buf);
    auto t4 = tnow();
    if (verbose)
        std::cout << "[b200] phases: cuda init " << secs(t0, t1) << " s, file read " << secs(t1, t2) << " s, hierarchy + upload + hot path + download "
                  << secs(t2, t3) << " s, plotfile write " << secs(t3, t4) << " s, kernels " << pa_kernel_launches() << "\n";
    return 0;
}
