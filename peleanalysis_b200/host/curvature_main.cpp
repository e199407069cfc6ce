// curvature3d.b200.ex -- drop-in for PeleAnalysis' curvature tool (R/Src/curvature.cpp): same ParmParse keys, plotfile
// in/out and output names; progress variable, flame normal, mean curvature and the optional Gaussian curvature /
// strain rate / normal velocity branches run through the C ABI.  do_smooth=1 (curvature.cpp:328-406) solves the implicit
// diffusion step with pa_smooth and runs the curvature on the smoothed field (one GPU only).  Extension: ngpus=N runs on N GPUs
// from this one process, one host thread per GPU (multi_gpu.hpp); transport=peer|slab picks peer links + packed slabs (default)
// or packed slabs only; smooth_precond=jacobi|mg picks do_smooth's preconditioner (default jacobi).
#include <algorithm>

#include "multi_gpu.hpp"
#include "tool_common.hpp"

int main(int argc, char** argv) {
    ParmParse pp(argc, argv);
    std::string progressName = "temp", plotFileName;
    double progMin = 1.0e20, progMax = -1.0e20, threshold = 0.0001, smooth_time = 1.0e-7;
    int finestLevel = 1000, verbose = 0, floorIt = 0, useFileMinMax = 1;
    bool do_strain = false, do_gaussCurv = false, getStrainTensor = false, do_velnormal = false, do_threshold = false, do_smooth = false;
    pp.query("verbose", verbose);
    pp.get("infile", plotFileName);
    std::string outfile = file_root(plotFileName) + "_K";
    pp.query("outfile", outfile);
    pp.query("finestLevel", finestLevel);
    pp.query("do_gaussCurv", do_gaussCurv);
    pp.query("progressName", progressName);
    pp.query("progMin", progMin);
    pp.query("progMax", progMax);
    pp.query("floorIt", floorIt);
    pp.query("useFileMinMax", useFileMinMax);
    pp.query("threshold_prog", do_threshold);
    pp.query("threshold_value", threshold);
    pp.query("do_smooth", do_smooth);
    pp.query("smoothing_time", smooth_time);
    std::string smooth_precond = "jacobi";
    pp.query("smooth_precond", smooth_precond);
    if (smooth_precond != "jacobi" && smooth_precond != "mg") pa_abort("smooth_precond must be jacobi or mg (got " + smooth_precond + ")");
    pp.query("do_strain", do_strain);
    if (do_strain) pp.query("getStrainTensor", getStrainTensor);
    pp.query("do_velnormal", do_velnormal);
    int nAux = pp.countval("Aux_Variables");
    std::vector<std::string> aux(nAux);
    for (int i = 0; i < nAux; ++i) pp.get("Aux_Variables", aux[i], i);

    std::cout << "infile = " << plotFileName << "\n" << "reading plt file = " << plotFileName << "\n";
    pltio::Header H;
    try { H = pltio::read_header(plotFileName); } catch (std::exception& e) { pa_abort(std::string("cannot read plotfile: ") + e.what()); }
    finestLevel = std::min(finestLevel, H.finest_level);
    const int Nlev = finestLevel + 1;
    const int idC = H.comp(progressName);
    if (idC < 0) pa_abort("Wrong progress variable name: " + progressName);
    if (useFileMinMax || floorIt) {
        if (useFileMinMax)
            for (int l = 0; l < Nlev; ++l) {                   // AmrData::MinMax over the whole domain = per-FAB header tables
                const auto& L = H.levels[l];
                if (L.fab_min.empty()) pa_abort("plotfile has no per-FAB min/max tables");
                for (size_t b = 0; b < L.boxes.size(); ++b) { progMin = std::min(progMin, L.fab_min[b][idC]); progMax = std::max(progMax, L.fab_max[b][idC]); }
            }
        std::cout << "progressName = " << progressName << " at index: " << idC << "\n" << "useFileMinMax = " << useFileMinMax << "\n"
                  << "Min/Max = " << progMin << " / " << progMax << "\n";
        if (progMin >= progMax) pa_abort("progMin must be less than progMax");
    }
    // variable index management (curvature.cpp:163-224)
    std::vector<std::string> inNames{progressName};
    // (the reference's idVst = 1: velocities follow the progress variable, curvature.cpp:172)
    if (do_strain) for (const char* v : {"x_velocity", "y_velocity", "z_velocity"}) inNames.push_back(v);
    for (auto& a : aux) { if (H.comp(a) < 0) pa_abort("Unknown auxiliary variable name: " + a); inNames.push_back(a); }
    const int nCompIn = (int)inNames.size();
    for (auto& n : inNames) if (H.comp(n) < 0) pa_abort("variable " + n + " not found in plotfile");
    const int idProg = nCompIn, idSmProg = idProg + 1, idKm = idSmProg + 1, idN = idKm + 1, idKg = idN + 3;
    int idSR = -1, nCompOut = idKg + 1;
    if (do_strain) { idSR = idKg + 1; nCompOut = idSR + 1; }
    int idROST = -1;
    if (getStrainTensor) { idROST = nCompOut; nCompOut += 9; }
    int idVelNormal = -1;
    if (do_velnormal) { idVelNormal = nCompOut; nCompOut += 1; }
    // the reference reads x/y/z_velocity only when do_strain is set; with do_velnormal alone it multiplies whatever sits
    // at idVst.. (curvature.cpp:772-774).  Here do_velnormal without do_strain reads the velocities explicitly.
    std::vector<std::string> velNames{"x_velocity", "y_velocity", "z_velocity"};
    const bool need_vel = do_strain || do_velnormal;
    if (need_vel) for (auto& v : velNames) if (H.comp(v) < 0) pa_abort("variable " + v + " not found in plotfile");

    std::vector<int> sym_dir(3, 0), is_per(3, 1);
    pp.queryarr("sym_dir", sym_dir, 0, 3);
    pp.queryarr("is_per", is_per, 0, 3);
    std::cout << "Periodicity assumed for this case: ";
    for (int d = 0; d < 3; ++d) std::cout << is_per[d] << " ";
    std::cout << "\n";

    int bck[3];
    for (int d = 0; d < 3; ++d) bck[d] = sym_dir[d] ? PA_BC_REFLECT_ODD : PA_BC_NEUMANN;
    pa_curv_opts o{};
    o.prog_min = progMin; o.prog_max = progMax; o.do_threshold = do_threshold; o.threshold = threshold;
    o.do_gauss = do_gaussCurv; o.do_strain = do_strain; o.get_strain_tensor = getStrainTensor; o.do_velnormal = do_velnormal;
    const int nres = pa_curvature_num_outputs(&o);
    // result component -> output slot, and the output names (curvature.cpp:794-829)
    std::vector<int> slot{idProg, idKm, idN, idN + 1, idN + 2};
    if (do_gaussCurv) slot.push_back(idKg);
    if (do_strain) slot.push_back(idSR);
    if (do_strain && getStrainTensor) for (int i = 0; i < 9; ++i) slot.push_back(idROST + i);
    if (do_velnormal) slot.push_back(idVelNormal);
    std::vector<std::string> names(nCompOut);
    for (int i = 0; i < nCompIn; ++i) names[i] = inNames[i];
    names[idProg] = "Progress"; names[idSmProg] = "SmoothedProgress"; names[idKm] = "MeanCurvature_" + progressName;
    names[idN] = "FlameNormalX_" + progressName; names[idN + 1] = "FlameNormalY_" + progressName; names[idN + 2] = "FlameNormalZ_" + progressName;
    names[idKg] = "GaussianCurvature_" + progressName;
    if (do_strain) names[idSR] = "StrainRate_" + progressName;
    if (getStrainTensor) {
        const char* dc[3] = {"x", "y", "z"};
        for (int i = 0; i < 9; ++i) names[idROST + i] = std::string("ROST_dU") + dc[i / 3] + "d" + dc[i % 3];
    }
    if (do_velnormal) names[idVelNormal] = "VelFlameNormal";
    // SmoothedProgress (do_smooth off) and GaussianCurvature (do_gaussCurv off) are never written by the reference
    // (uninitialised memory there); they are written as zeros here.
    std::vector<int> zero_slots;
    if (!do_smooth) zero_slots.push_back(idSmProg);
    if (!do_gaussCurv) zero_slots.push_back(idKg);
    if (getStrainTensor && !do_strain) for (int i = 0; i < 9; ++i) zero_slots.push_back(idROST + i);

    int ngpus = 1;
    pp.query("ngpus", ngpus);
    std::string transport = "peer";
    pp.query("transport", transport);
    if (transport != "peer" && transport != "slab") pa_abort("transport must be peer or slab (got " + transport + ")");
    if (ngpus > 1 && do_smooth)
        pa_abort("do_smooth=1 runs on one GPU only: the smoothing solve has no multi-GPU path (use ngpus=1)");
    if (ngpus > 1) {
        CurvJob J;
        J.peer = transport == "peer";
        J.verbose = verbose != 0;
        J.infile = plotFileName; J.outfile = outfile; J.H = &H; J.Nlev = Nlev;
        J.inNames = inNames; J.velNames = velNames; J.names = names; J.need_vel = need_vel; J.o = o;
        J.slot = slot; J.zero_slots = zero_slots; J.nCompOut = nCompOut; J.is_per = is_per;
        for (int d = 0; d < 3; ++d) J.bck[d] = bck[d];
        std::cout << "Writing new data to " << outfile << "\n";
        run_curv_multi(ngpus, J);
        return 0;
    }

    check(pa_init(0), "pa_init");
    HierInput hi;
    make_level_descs(H, Nlev, hi);
    pa_hier* h = nullptr;
    check(pa_hier_create(&h, Nlev, hi.lv.data(), is_per.data(), bck, 0, 1), "pa_hier_create");
    pa_field *st = nullptr, *res = nullptr;
    // do_smooth: two more state components, c and the smoothed phi, which the curvature then reads as its scalar
    const int nst = need_vel ? 4 : 1, comp_c = nst, comp_phi = nst + 1;
    check(pa_field_alloc(h, do_smooth ? nst + 2 : nst, 1, &st), "pa_field_alloc");
    check(pa_field_alloc(h, nres, 1, &res), "pa_field_alloc");

    std::vector<PinnedLevel> buf(Nlev);
    std::vector<PinnedLevel> velbuf(Nlev);
    for (int l = 0; l < Nlev; ++l) {
        if (verbose) std::cout << "Reading data for level " << l << "\n";
        buf[l].alloc(H.levels[l].ncells(), nCompOut);
        for (int c = 0; c < nCompIn; ++c) pltio::read_level_comp(plotFileName, H, l, H.comp(inNames[c]), buf[l].comp(c));
        check(pa_field_upload_level(st, l, 0, buf[l].comp(0)), "upload");
        if (need_vel) {
            velbuf[l].alloc(H.levels[l].ncells(), 3);
            for (int d = 0; d < 3; ++d) {
                pltio::read_level_comp(plotFileName, H, l, H.comp(velNames[d]), velbuf[l].comp(d));
                check(pa_field_upload_level(st, l, 1 + d, velbuf[l].comp(d)), "upload");
            }
        }
    }
    if (do_smooth) {
        pa_smooth_opts so{};
        so.smoothing_time = smooth_time;
        so.precond = smooth_precond == "mg" ? PA_SMOOTH_PRECOND_MG : PA_SMOOTH_PRECOND_JACOBI;
        int iters = 0;
        double resid = 0.0;
        check(pa_smooth(st, 0, progMin, progMax, &so, st, comp_c, comp_phi, &iters, &resid), "pa_smooth");
        if (verbose) std::cout << "do_smooth: smoothing_time = " << smooth_time << ", precond " << smooth_precond << ", " << iters
                               << " iterations, max|c - A phi| / max|c| = " << resid << "\n";
        // the curvature of phi with the identity normalisation (curvature.cpp:328-406 hands the solution on as the progress
        // variable); its Progress output is phi itself and goes to SmoothedProgress, Progress is c
        pa_curv_opts os = o;
        os.prog_min = 0.0; os.prog_max = 1.0;
        slot[0] = idSmProg;
        check(pa_curvature(st, comp_phi, 1, &os, res, 0), "pa_curvature");
    } else {
        check(pa_curvature(st, 0, 1, &o, res, 0), "pa_curvature");
    }
    {
        long long mx = 0;
        for (int l = 0; l < Nlev; ++l) mx = std::max(mx, buf[l].ncells);
        StagedDownloader dl(mx);
        for (int l = 0; l < Nlev; ++l) {
            for (int z : zero_slots) std::fill(buf[l].comp(z), buf[l].comp(z) + buf[l].ncells, 0.0);
            for (int c = 0; c < nres; ++c) dl.download(res, l, c, buf[l].comp(slot[c]), buf[l].ncells);
            if (do_smooth) dl.download(st, l, comp_c, buf[l].comp(idProg), buf[l].ncells);
        }
        dl.flush();
    }
    check(pa_sync(), "pa_sync");

    std::cout << "Writing new data to " << outfile << "\n";
    std::vector<std::vector<const double*>> data(Nlev);
    for (int l = 0; l < Nlev; ++l) for (int c = 0; c < nCompOut; ++c) data[l].push_back(buf[l].comp(c));
    std::vector<int> rr(std::max(Nlev - 1, 0), 2);            // curvature.cpp:842
    pltio::Header meta = H;
    meta.time = 0.0;
    try { pltio::write_plotfile(outfile, meta, names, data, rr); } catch (std::exception& e) { pa_abort(e.what()); }
    pa_field_free(st); pa_field_free(res); pa_hier_destroy(h);
    return 0;
}
