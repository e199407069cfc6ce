// curvature3d.b200.ex -- drop-in for PeleAnalysis' curvature tool (R/Src/curvature.cpp): same ParmParse keys, plotfile
// in/out and output names; progress variable, flame normal, mean curvature and the optional Gaussian curvature /
// strain rate / normal velocity branches run through the C ABI.  do_smooth=1 (curvature.cpp:328-406) solves the implicit
// diffusion step with pa_smooth and runs the curvature on the smoothed field (one GPU only).  Extension: ngpus=N runs on N GPUs
// from this one process, one host thread per GPU (multi_gpu.hpp); transport=peer|slab picks peer links + packed slabs (default)
// or packed slabs only; smooth_precond=jacobi|mg picks do_smooth's preconditioner (default jacobi); infiles=a b c runs a
// series of plotfiles in one process (series.hpp), every other key applying to each file.
#include <algorithm>

#include "multi_gpu.hpp"
#include "series.hpp"

struct CurvKeys {                                      // the keys every file of a run shares
    std::string progressName = "temp", smooth_precond = "jacobi";
    double progMin = 1.0e20, progMax = -1.0e20, threshold = 0.0001, smooth_time = 1.0e-7;
    int finestLevel = 1000, floorIt = 0, useFileMinMax = 1;
    bool do_strain = false, do_gaussCurv = false, getStrainTensor = false, do_velnormal = false, do_threshold = false, do_smooth = false;
    std::vector<std::string> aux;
    std::vector<int> is_per;
    int bck[3];
};

struct CurvFile {                                      // one plotfile, checked: its inputs, output slots and names
    std::string infile, outfile;
    pltio::Header H, meta;                             // the plotfile; the output's header (time 0)
    int Nlev = 0;
    std::vector<std::string> inNames, velNames{"x_velocity", "y_velocity", "z_velocity"}, names;
    bool need_vel = false;
    pa_curv_opts o{};
    int nCompIn = 0, nCompOut = 0, idProg = 0, idSmProg = 0, nres = 0;
    std::vector<int> slot, zero_slots;
};

// the checks of a single run on one plotfile; `who` prefixes every abort message (a series names the file)
static CurvFile curv_file(const CurvKeys& k, const std::string& infile, const std::string& who, bool talk) {
    CurvFile F;
    F.infile = infile;
    F.outfile = file_root(infile) + "_K";
    if (talk) std::cout << "infile = " << infile << "\n" << "reading plt file = " << infile << "\n";
    const pltio::Header& H = F.H;
    try { F.H = pltio::read_header(infile); } catch (std::exception& e) { pa_abort(who + std::string("cannot read plotfile: ") + e.what()); }
    F.Nlev = std::min(k.finestLevel, H.finest_level) + 1;
    const int Nlev = F.Nlev;
    const int idC = H.comp(k.progressName);
    if (idC < 0) pa_abort(who + "Wrong progress variable name: " + k.progressName);
    double progMin = k.progMin, progMax = k.progMax;
    if (k.useFileMinMax || k.floorIt) {
        if (k.useFileMinMax)
            for (int l = 0; l < Nlev; ++l) {                   // AmrData::MinMax over the whole domain = per-FAB header tables
                const auto& L = H.levels[l];
                if (L.fab_min.empty()) pa_abort(who + "plotfile has no per-FAB min/max tables");
                for (size_t b = 0; b < L.boxes.size(); ++b) { progMin = std::min(progMin, L.fab_min[b][idC]); progMax = std::max(progMax, L.fab_max[b][idC]); }
            }
        if (talk)
            std::cout << "progressName = " << k.progressName << " at index: " << idC << "\n" << "useFileMinMax = " << k.useFileMinMax << "\n"
                      << "Min/Max = " << progMin << " / " << progMax << "\n";
        if (progMin >= progMax) pa_abort(who + "progMin must be less than progMax");
    }
    // variable index management (curvature.cpp:163-224)
    F.inNames.push_back(k.progressName);
    // (the reference's idVst = 1: velocities follow the progress variable, curvature.cpp:172)
    if (k.do_strain) for (const char* v : {"x_velocity", "y_velocity", "z_velocity"}) F.inNames.push_back(v);
    for (auto& a : k.aux) { if (H.comp(a) < 0) pa_abort(who + "Unknown auxiliary variable name: " + a); F.inNames.push_back(a); }
    const int nCompIn = F.nCompIn = (int)F.inNames.size();
    for (auto& n : F.inNames) if (H.comp(n) < 0) pa_abort(who + "variable " + n + " not found in plotfile");
    const int idProg = nCompIn, idSmProg = idProg + 1, idKm = idSmProg + 1, idN = idKm + 1, idKg = idN + 3;
    F.idProg = idProg; F.idSmProg = idSmProg;
    int idSR = -1, nCompOut = idKg + 1;
    if (k.do_strain) { idSR = idKg + 1; nCompOut = idSR + 1; }
    int idROST = -1;
    if (k.getStrainTensor) { idROST = nCompOut; nCompOut += 9; }
    int idVelNormal = -1;
    if (k.do_velnormal) { idVelNormal = nCompOut; nCompOut += 1; }
    F.nCompOut = nCompOut;
    // the reference reads x/y/z_velocity only when do_strain is set; with do_velnormal alone it multiplies whatever sits
    // at idVst.. (curvature.cpp:772-774).  Here do_velnormal without do_strain reads the velocities explicitly.
    F.need_vel = k.do_strain || k.do_velnormal;
    if (F.need_vel) for (auto& v : F.velNames) if (H.comp(v) < 0) pa_abort(who + "variable " + v + " not found in plotfile");

    pa_curv_opts& o = F.o;
    o.prog_min = progMin; o.prog_max = progMax; o.do_threshold = k.do_threshold; o.threshold = k.threshold;
    o.do_gauss = k.do_gaussCurv; o.do_strain = k.do_strain; o.get_strain_tensor = k.getStrainTensor; o.do_velnormal = k.do_velnormal;
    F.nres = pa_curvature_num_outputs(&o);
    // result component -> output slot, and the output names (curvature.cpp:794-829)
    F.slot = {idProg, idKm, idN, idN + 1, idN + 2};
    if (k.do_gaussCurv) F.slot.push_back(idKg);
    if (k.do_strain) F.slot.push_back(idSR);
    if (k.do_strain && k.getStrainTensor) for (int i = 0; i < 9; ++i) F.slot.push_back(idROST + i);
    if (k.do_velnormal) F.slot.push_back(idVelNormal);
    std::vector<std::string>& names = F.names;
    names.resize(nCompOut);
    const std::string& progressName = k.progressName;
    for (int i = 0; i < nCompIn; ++i) names[i] = F.inNames[i];
    names[idProg] = "Progress"; names[idSmProg] = "SmoothedProgress"; names[idKm] = "MeanCurvature_" + progressName;
    names[idN] = "FlameNormalX_" + progressName; names[idN + 1] = "FlameNormalY_" + progressName; names[idN + 2] = "FlameNormalZ_" + progressName;
    names[idKg] = "GaussianCurvature_" + progressName;
    if (k.do_strain) names[idSR] = "StrainRate_" + progressName;
    if (k.getStrainTensor) {
        const char* dc[3] = {"x", "y", "z"};
        for (int i = 0; i < 9; ++i) names[idROST + i] = std::string("ROST_dU") + dc[i / 3] + "d" + dc[i % 3];
    }
    if (k.do_velnormal) names[idVelNormal] = "VelFlameNormal";
    // SmoothedProgress (do_smooth off) and GaussianCurvature (do_gaussCurv off) are never written by the reference
    // (uninitialised memory there); they are written as zeros here.
    if (!k.do_smooth) F.zero_slots.push_back(idSmProg);
    if (!k.do_gaussCurv) F.zero_slots.push_back(idKg);
    if (k.getStrainTensor && !k.do_strain) for (int i = 0; i < 9; ++i) F.zero_slots.push_back(idROST + i);
    F.meta = H;
    F.meta.time = 0.0;
    return F;
}

// disk -> in[l] of the rank's boxes: components 0 .. nCompIn-1 the pass-through inputs (progress variable first); in_place:
// room for the results as well; with velocities, three more components last
static void curv_read(const CurvFile& F, const RankCtx& R, HostSet& in, bool in_place, bool talk) {
    ensure_levels(in, F.Nlev);
    const int nalloc = (in_place ? F.nCompOut : F.nCompIn) + (F.need_vel ? 3 : 0);
    for (int l = 0; l < F.Nlev; ++l) {
        if (talk) std::cout << "Reading data for level " << l << "\n";
        in[l].alloc(R.cells(F.H, l), nalloc);
        for (int c = 0; c < F.nCompIn; ++c) pltio::read_boxes_comp(F.infile, F.H, l, F.H.comp(F.inNames[c]), R.mine[l], in[l].comp(c));
        if (F.need_vel)
            for (int d = 0; d < 3; ++d) pltio::read_boxes_comp(F.infile, F.H, l, F.H.comp(F.velNames[d]), R.mine[l], in[l].comp(nalloc - 3 + d));
    }
}

static void curv_gpu(const CurvKeys& k, const CurvFile& F, const RankCtx& R, HostSet& in, HostSet& out, StagedDownloader& dl, bool talk) {
    const int Nlev = F.Nlev, nres = F.nres;
    pa_hier* h = R.hier(F.H, Nlev, k.is_per.data(), k.bck, 0);
    pa_field *st = nullptr, *res = nullptr, *scratch = nullptr;
    // do_smooth: two more state components, c and the smoothed phi, which the curvature then reads as its scalar
    const int nst = F.need_vel ? 4 : 1, comp_c = nst, comp_phi = nst + 1;
    check(pa_field_alloc(h, k.do_smooth ? nst + 2 : nst, 1, &st), "pa_field_alloc");
    check(pa_field_alloc(h, nres, 1, &res), "pa_field_alloc");
    if (F.o.do_gauss) check(pa_curvature_scratch(h, 0, &scratch), "pa_curvature_scratch");
    for (int l = 0; l < Nlev; ++l) {
        check(pa_field_upload_level(st, l, 0, in[l].comp(0)), "upload");
        if (F.need_vel)
            for (int d = 0; d < 3; ++d) check(pa_field_upload_level(st, l, 1 + d, in[l].comp(in[l].ncomp - 3 + d)), "upload");
    }
    std::vector<pa_field*> fields{st, res};
    if (scratch) fields.push_back(scratch);
    R.map_peers(Nlev, fields);
    std::vector<int> slot = F.slot;
    pa_curv_opts o = F.o;
    int comp_S = 0;
    if (k.do_smooth) {
        pa_smooth_opts so{};
        so.smoothing_time = k.smooth_time;
        so.precond = k.smooth_precond == "mg" ? PA_SMOOTH_PRECOND_MG : PA_SMOOTH_PRECOND_JACOBI;
        int iters = 0;
        double resid = 0.0;
        check(pa_smooth(st, 0, F.o.prog_min, F.o.prog_max, &so, st, comp_c, comp_phi, &iters, &resid), "pa_smooth");
        if (talk) std::cout << "do_smooth: smoothing_time = " << k.smooth_time << ", precond " << k.smooth_precond << ", " << iters
                            << " iterations, max|c - A phi| / max|c| = " << resid << "\n";
        // the curvature of phi with the identity normalisation (curvature.cpp:328-406 hands the solution on as the progress
        // variable); its Progress output is phi itself and goes to SmoothedProgress, Progress is c
        o.prog_min = 0.0; o.prog_max = 1.0;
        slot[0] = F.idSmProg;
        comp_S = comp_phi;
    }
    // the steps of pa_curvature, each behind the cross-rank step it needs
    auto step = [&](int steps, int lev) { check(pa_curvature_steps(st, comp_S, 1, &o, res, 0, steps, lev, lev), "pa_curvature"); };
    R.exchange(st, comp_S, 1);
    step(PA_CURV_PASS1, -1);
    if (o.do_threshold) {
        for (int l = 0; l < Nlev; ++l) {
            R.exchange(res, 2, 3);
            step(PA_CURV_DIV, l);
            // the clip zeroes n(l) in place; with peer links every rank's DIV(l) reads its peers' UNCLIPPED n(l) over the links
            // first (curvature.cpp:487-567: FillBoundary of n precedes the clip).  With transport=slab the peers' cells of n(l)
            // were copied inside the exchange, which ends in a barrier: nothing reads n(l) in place.
            if (R.peer_links) {
                check(pa_sync(), "pa_sync");
                R.barrier();
            }
            step(PA_CURV_CLIP, l);
        }
    } else {
        R.exchange(res, 2, 3);
        step(PA_CURV_DIV, -1);
    }
    if (o.do_gauss) { R.exchange(scratch, 0, 3); step(PA_CURV_GAUSS, -1); }
    if (o.do_strain) { R.exchange(st, 1, 3); step(PA_CURV_STRAIN, -1); }
    if (o.do_velnormal) step(PA_CURV_VELN, -1);

    ensure_levels(out, Nlev);
    long long mx = 0;
    for (int l = 0; l < Nlev; ++l) {
        const long long nc = in[l].ncells;
        mx = std::max(mx, nc);
        if (&out != &in) {
            out[l].alloc(nc, F.nCompOut);
            std::memcpy(out[l].comp(0), in[l].comp(0), (size_t)F.nCompIn * nc * 8);
        }
    }
    dl.reserve(mx);
    for (int l = 0; l < Nlev; ++l) {
        PinnedLevel& b = out[l];
        for (int z : F.zero_slots) std::fill(b.comp(z), b.comp(z) + b.ncells, 0.0);
        for (int c = 0; c < nres; ++c) dl.download(res, l, c, b.comp(slot[c]), b.ncells);
        if (k.do_smooth) dl.download(st, l, comp_c, b.comp(F.idProg), b.ncells);
    }
    dl.flush();
    check(pa_sync(), "pa_sync");
    R.barrier();                                       // nobody frees a slab a peer may still be reading
    pa_field_free(st); pa_field_free(res); pa_hier_destroy(h);
}

int main(int argc, char** argv) {
    ParmParse pp(argc, argv);
    CurvKeys k;
    int verbose = 0;
    pp.query("verbose", verbose);
    const bool series = pp.contains("infiles");
    std::vector<std::string> infiles;
    std::string plotFileName, outfile;
    if (series) infiles = series_inputs(pp);
    else pp.get("infile", plotFileName);
    pp.query("outfile", outfile);
    pp.query("finestLevel", k.finestLevel);
    pp.query("do_gaussCurv", k.do_gaussCurv);
    pp.query("progressName", k.progressName);
    pp.query("progMin", k.progMin);
    pp.query("progMax", k.progMax);
    pp.query("floorIt", k.floorIt);
    pp.query("useFileMinMax", k.useFileMinMax);
    pp.query("threshold_prog", k.do_threshold);
    pp.query("threshold_value", k.threshold);
    pp.query("do_smooth", k.do_smooth);
    pp.query("smoothing_time", k.smooth_time);
    pp.query("smooth_precond", k.smooth_precond);
    if (k.smooth_precond != "jacobi" && k.smooth_precond != "mg") pa_abort("smooth_precond must be jacobi or mg (got " + k.smooth_precond + ")");
    pp.query("do_strain", k.do_strain);
    if (k.do_strain) pp.query("getStrainTensor", k.getStrainTensor);
    pp.query("do_velnormal", k.do_velnormal);
    k.aux.resize(pp.countval("Aux_Variables"));
    for (size_t i = 0; i < k.aux.size(); ++i) pp.get("Aux_Variables", k.aux[i], (int)i);
    std::vector<int> sym_dir(3, 0);
    k.is_per.assign(3, 1);
    pp.queryarr("sym_dir", sym_dir, 0, 3);
    pp.queryarr("is_per", k.is_per, 0, 3);
    for (int d = 0; d < 3; ++d) k.bck[d] = sym_dir[d] ? PA_BC_REFLECT_ODD : PA_BC_NEUMANN;
    int ngpus = 1;
    pp.query("ngpus", ngpus);

    // the threads of ngpus=N and the files of a series print no progress lines
    ToolBody<CurvFile> body;
    body.read = [&](const CurvFile& F, const RankCtx& R, HostSet& in, bool in_place) { curv_read(F, R, in, in_place, false); };
    body.gpu = [&](const CurvFile& F, const RankCtx& R, HostSet& in, HostSet& out, StagedDownloader& dl) { curv_gpu(k, F, R, in, out, dl, false); };

    if (series) {
        // every header read and checked before anything is computed or written; each file runs on one GPU, so do_smooth too
        std::vector<CurvFile> files;
        for (auto& f : infiles) files.push_back(curv_file(k, f, f + ": ", false));
        check_distinct_outputs(files);
        run_series(ngpus, files, body, verbose != 0);
        return 0;
    }

    CurvFile F = curv_file(k, plotFileName, "", true);
    if (!outfile.empty()) F.outfile = outfile;
    std::cout << "Periodicity assumed for this case: ";
    for (int d = 0; d < 3; ++d) std::cout << k.is_per[d] << " ";
    std::cout << "\n";

    std::string transport = "peer";
    pp.query("transport", transport);
    if (transport != "peer" && transport != "slab") pa_abort("transport must be peer or slab (got " + transport + ")");
    if (ngpus > 1 && k.do_smooth)
        pa_abort("do_smooth=1 runs on one GPU only: the smoothing solve has no multi-GPU path (use ngpus=1)");
    if (ngpus > 1) {
        std::cout << "Writing new data to " << F.outfile << "\n";
        run_ranks(ngpus, F, body, transport == "peer", verbose != 0);
        return 0;
    }

    check(pa_init(0), "pa_init");
    const RankCtx R(F.meta, F.Nlev);
    // one buffer set holds the inputs and receives the results
    HostSet buf;
    curv_read(F, R, buf, true, verbose != 0);
    {
        StagedDownloader dl(0);
        curv_gpu(k, F, R, buf, buf, dl, verbose != 0);
    }
    std::cout << "Writing new data to " << F.outfile << "\n";
    R.write(F, buf);
    return 0;
}
