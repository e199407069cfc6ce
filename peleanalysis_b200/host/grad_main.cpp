// grad3d.b200.ex -- drop-in for PeleAnalysis' grad tool (R/Src/grad.cpp): same ParmParse keys, same plotfile in/out,
// same output variable names; the operator block (grad.cpp:151-236) is the C ABI of libpelestencil_b200.
//
//   grad3d.b200.ex infile=<plotfile> [gradVar=temp] [finestLevel=N] [Aux_Variables=a b ...] [is_per=1 1 1]
//                  [sym_dir=0 0 0] [outfile=<name>]          extensions: gradVars=a b c  (several variables, one pass)
//                                                                        ngpus=N  (one host thread per GPU, multi_gpu.hpp)
//                                                                        transport=peer|slab  (with ngpus=N: peer links +
//                                                                        packed slabs, or packed slabs only)
#include <chrono>

#include "multi_gpu.hpp"
#include "tool_common.hpp"

static void print_usage(char** argv) {
    std::cerr << "usage:\n" << argv[0] << " infile=<plotfilename> \n\tOptions:\n\tis_per=<L M N> gradVar=<name>\n";
    std::exit(1);
}

int main(int argc, char** argv) {
    if (argc < 2) print_usage(argv);
    ParmParse pp(argc, argv);
    if (pp.contains("help")) print_usage(argv);
    std::string infile, gradVar = "temp";
    int finestLevel = 1000, verbose = 0;
    pp.get("infile", infile);
    pp.query("gradVar", gradVar);
    pp.query("finestLevel", finestLevel);
    pp.query("verbose", verbose);

    pltio::Header H;
    try { H = pltio::read_header(infile); } catch (std::exception& e) { pa_abort(std::string("cannot read plotfile: ") + e.what()); }
    finestLevel = std::min(finestLevel, H.finest_level);
    const int Nlev = finestLevel + 1;

    std::vector<std::string> gvars;
    int ng = pp.countval("gradVars");
    if (ng > 0) { gvars.resize(ng); for (int i = 0; i < ng; ++i) pp.get("gradVars", gvars[i], i); }
    else gvars.push_back(gradVar);
    for (auto& v : gvars)
        if (H.comp(v) < 0) { std::cout << "Cannot find " << v << " data in pltfile \n"; pa_abort("Cannot find " + v + " data in pltfile"); }
    int nAux = pp.countval("Aux_Variables");
    std::vector<std::string> aux(nAux);
    for (int i = 0; i < nAux; ++i) {
        pp.get("Aux_Variables", aux[i], i);
        if (H.comp(aux[i]) < 0) pa_abort("Unknown auxiliary variable name: " + aux[i]);
    }
    std::vector<int> sym_dir(3, 0), is_per(3, 1);
    pp.queryarr("sym_dir", sym_dir, 0, 3);
    pp.queryarr("is_per", is_per, 0, 3);
    std::cout << "Periodicity assumed for this case: ";
    for (int d = 0; d < 3; ++d) std::cout << is_per[d] << " ";
    std::cout << "\n";

    int ngpus = 1;
    pp.query("ngpus", ngpus);
    std::string transport = "peer";
    pp.query("transport", transport);
    if (transport != "peer" && transport != "slab") pa_abort("transport must be peer or slab (got " + transport + ")");
    if (ngpus > 1) {
        GradJob J;
        J.infile = infile; J.H = &H; J.Nlev = Nlev; J.gvars = gvars; J.aux = aux; J.is_per = is_per;
        J.peer = transport == "peer";
        J.verbose = verbose != 0;
        for (int d = 0; d < 3; ++d) J.bck[d] = sym_dir[d] ? PA_BC_REFLECT_ODD : PA_BC_NEUMANN;
        for (auto& v : gvars) J.names.push_back(v);
        for (auto& a : aux) J.names.push_back(a);
        for (auto& v : gvars) { J.names.push_back(v + "_gx"); J.names.push_back(v + "_gy"); J.names.push_back(v + "_gz"); J.names.push_back("||grad" + v + "||"); }
        J.outfile = file_root(infile) + "_gt";
        pp.query("outfile", J.outfile);
        std::cout << "Writing new data to " << J.outfile << std::endl;
        run_grad_multi(ngpus, J);
        return 0;
    }
    auto t0 = std::chrono::steady_clock::now();
    auto tnow = [] { return std::chrono::steady_clock::now(); };
    auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
    double t_init = 0, t_pin = 0, t_read = 0;
    check(pa_init(0), "pa_init");
    t_init = secs(t0, tnow());
    HierInput hi;
    make_level_descs(H, Nlev, hi);
    int bck[3];
    for (int d = 0; d < 3; ++d) bck[d] = sym_dir[d] ? PA_BC_REFLECT_ODD : PA_BC_NEUMANN;
    pa_hier* h = nullptr;
    check(pa_hier_create(&h, Nlev, hi.lv.data(), is_per.data(), bck, 0, 1), "pa_hier_create");
    const int nv = (int)gvars.size();
    pa_field *fin = nullptr, *fout = nullptr;
    check(pa_field_alloc(h, nv, 1, &fin), "pa_field_alloc");
    check(pa_field_alloc(h, 4 * nv, 0, &fout), "pa_field_alloc");

    // read: gradient variables go to the device, pass-through variables stay on the host
    const int nIn = nv + nAux, nOut = nIn + 4 * nv;
    std::vector<PinnedLevel> buf(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        std::cout << "Reading data for level: " << l << std::endl;
        auto ta = tnow();
        buf[l].alloc(H.levels[l].ncells(), nOut);
        auto tb = tnow();
        for (int v = 0; v < nv; ++v) {
            pltio::read_level_comp(infile, H, l, H.comp(gvars[v]), buf[l].comp(v));
            check(pa_field_upload_level(fin, l, v, buf[l].comp(v)), "upload");
        }
        for (int a = 0; a < nAux; ++a) pltio::read_level_comp(infile, H, l, H.comp(aux[a]), buf[l].comp(nv + a));
        t_pin += secs(ta, tb); t_read += secs(tb, tnow());
    }
    auto t1 = std::chrono::steady_clock::now();
    check(pa_grad(fin, 0, nv, fout, 0), "pa_grad");
    {
        long long mx = 0;
        for (int l = 0; l < Nlev; ++l) mx = std::max(mx, H.levels[l].ncells());
        StagedDownloader dl(mx);
        for (int l = 0; l < Nlev; ++l)
            for (int c = 0; c < 4 * nv; ++c) dl.download(fout, l, c, buf[l].comp(nIn + c), H.levels[l].ncells());
        dl.flush();
    }
    check(pa_sync(), "pa_sync");
    auto t2 = std::chrono::steady_clock::now();

    std::vector<std::string> names;
    for (auto& v : gvars) names.push_back(v);
    for (auto& a : aux) names.push_back(a);
    for (auto& v : gvars) { names.push_back(v + "_gx"); names.push_back(v + "_gy"); names.push_back(v + "_gz"); names.push_back("||grad" + v + "||"); }
    std::string outfile = file_root(infile) + "_gt";
    pp.query("outfile", outfile);
    std::cout << "Writing new data to " << outfile << std::endl;
    std::vector<std::vector<const double*>> data(Nlev);
    for (int l = 0; l < Nlev; ++l) for (int c = 0; c < nOut; ++c) data[l].push_back(buf[l].comp(c));
    std::vector<int> rr(std::max(Nlev - 1, 0), 2);            // the reference hard-codes refRatios = 2 (grad.cpp:255)
    pltio::Header meta = H;
    meta.time = 0.0;                                           // WriteMultiLevelPlotfile(..., 0.0, ...) (grad.cpp:256)
    try { pltio::write_plotfile(outfile, meta, names, data, rr); } catch (std::exception& e) { pa_abort(e.what()); }
    auto t3 = tnow();
    if (verbose) {
        auto s = [](auto a, auto b) { return std::chrono::duration<double>(b - a).count(); };
        std::cout << "[b200] read+upload " << s(t0, t1) << " s, hot path+download " << s(t1, t2) << " s, kernels " << pa_kernel_launches() << "\n";
        std::cout << "[b200] phases: cuda init " << t_init << " s, pinned alloc " << t_pin << " s, file read + upload " << t_read
                  << " s, hierarchy + fields " << s(t0, t1) - t_init - t_pin - t_read << " s, plotfile write " << s(t2, t3) << " s\n";
    }
    pa_field_free(fin); pa_field_free(fout); pa_hier_destroy(h);
    return 0;
}
