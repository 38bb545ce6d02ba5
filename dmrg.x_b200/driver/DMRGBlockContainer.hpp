/*  DMRGBlockContainer — host mirror of include/DMRGBlockContainer.hpp:166-2765 over the C ABI.
 *
 *  Same public surface (Initialize, SetUpCorrelation, Warmup, Sweeps, SingleSweep, Destroy, SysBlock, NumSites,
 *  Verbose, HamiltonianRef), same option names, same schedule of SingleDMRGStep calls and the same JSON
 *  outputs (DMRGSteps.json, Timings.json, EntanglementSpectra.json, DMRGRun.json, Correlations.json).
 *  What changes is where the work happens: every phase of SingleDMRGStep is one C-ABI call into the sm_100a
 *  library, blocks stay resident in HBM between steps (the reference's scratch-disk round trips are no-ops), and
 *  the SLEPc EPS object becomes dmrgx_eigs_smallest with the `-H_eps_*` options.
 */
#pragma once
#include <unistd.h>
#include <algorithm>
#include <chrono>
#include <cmath>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <memory>
#include <set>

#include "DMRGBlockIO.hpp"
#include "DMRGKron.hpp"

/** include/DMRGBlockContainer.hpp:21-27 */
typedef enum { BlockSys = 0, BlockEnv = 1 } Block_t;
/** include/DMRGBlockContainer.hpp:30-35 */
struct Op { Op_t OpType; PetscInt idx; };
inline std::string OpToStr(const Op_t& OpType) {
    switch (OpType) { case OpSm: return "Sm"; case OpSz: return "Sz"; case OpSp: return "Sp"; case OpEye: return "Eye"; }
    return "";
}
/** include/DMRGBlockContainer.hpp:40-80 */
struct Correlator {
    PetscInt idx = 0;
    std::vector<Op> SysOps, EnvOps;
    std::string name, desc1, desc2, desc3;
};

/** BasisTransformation (include/DMRGBlockContainer.hpp:226-257): RotMatT stays on the device behind the handle */
struct BasisTransformation {
    dmrgx_xform h = nullptr;
    QuantumNumbers QN;
    PetscReal TruncErr = 0;
    PetscInt m = 0;
    ~BasisTransformation() { if (h) dmrgx_xform_destroy(h); }
    PetscErrorCode Load() {
        dmrgx_int mm, n, ns, ne;
        DMRGX_CALL(dmrgx_xform_info(h, &mm, &n, &ns, &TruncErr, &ne));
        m = mm;
        std::vector<PetscReal> qn((size_t)ns); std::vector<PetscInt> sz((size_t)ns);
        DMRGX_CALL(dmrgx_xform_sectors(h, qn.data(), sz.data()));
        return QN.Initialize(0, qn, sz);
    }
};

template <class Block, class Hamiltonian>
class DMRGBlockContainer {
public:
    explicit DMRGBlockContainer(const MPI_Comm& mpi_comm) : mpi_comm(mpi_comm) {}
    ~DMRGBlockContainer() { Destroy(); }

    /** :272-587 */
    PetscErrorCode Initialize() {
        if (init) SETERRQ(mpi_comm, 1, "DMRG object has already been initialized.");
        PetscOptions& o = PetscOptions::DB();
        PetscErrorCode ierr;
        std::string path; PetscBool set = PETSC_FALSE;
        /* -restart_dir: the directory of a previous run's scratch; continue from its last Sweep_* with a valid Sweep.dat (:286-347) */
        o.GetString("-restart_dir", path, &restart);
        if (restart) {
            restart_dir = path;
            if (restart_dir.back() != '/') restart_dir += "/";
            PetscInt ridx = 0;
            auto exists = [](const std::string& f) { std::ifstream t(f.c_str()); return (bool)t; };
            while (ridx < MAX_SWEEP_IDX && !exists(restart_dir + SweepDir(ridx) + "Sweep.dat")) ++ridx;
            if (ridx == MAX_SWEEP_IDX) SETERRQ1(mpi_comm, 1, "No Sweep directory was found in %s", restart_dir.c_str());
            while (ridx < MAX_SWEEP_IDX && exists(restart_dir + SweepDir(ridx + 1) + "Sweep.dat")) ++ridx;
            restart_dir = restart_dir + SweepDir(ridx);
            { /* the Hamiltonian of the previous run (Hamiltonian.dat is an options file) */
                std::ifstream in((restart_dir + "Hamiltonian.dat").c_str());
                if (!in) SETERRQ1(mpi_comm, 1, "cannot read %sHamiltonian.dat", restart_dir.c_str());
                std::stringstream ss; ss << in.rdbuf();
                o.InsertString(ss.str());
            }
            /* the spin type of the saved blocks rules the sites added from now on (src/DMRGBlock.cpp:280-315): a conflicting -spin
               is an error, a missing one is imposed — before SingleSite is created below */
            ierr = BlockIO::ApplySpinTypeOfBlockDir(restart_dir + BlockDir("Sys", 0)); CHKERRQ(ierr);
            std::map<std::string, PetscInt> d;
            { std::ifstream in((restart_dir + "Sweep.dat").c_str()); for (std::string k; in >> k;) { PetscInt v; in >> v; d[k] = v; } }
            for (const char* k : {"GlobIdx", "LoopIdx", "num_sys_blocks", "sys_ninit"}) if (!d.count(k)) SETERRQ1(mpi_comm, 1, "Sweep.dat: %s not found.", k);
            GlobIdx = d["GlobIdx"]; LoopIdx = d["LoopIdx"] + 1; num_sys_blocks = d["num_sys_blocks"]; sys_ninit = d["sys_ninit"];
            std::cout << "WARNING:\nThe following variables have been forcefully set:\n  GlobIdx " << GlobIdx << "\n  LoopIdx " << LoopIdx
                      << "\n  num_sys_blocks " << num_sys_blocks << "\n  sys_ninit " << sys_ninit << std::endl;
        }

        ierr = Ham.SetFromOptions(); CHKERRQ(ierr);
        ierr = SingleSite.Initialize(mpi_comm, 1, PETSC_DEFAULT); CHKERRQ(ierr);
        num_sites = Ham.NumSites();
        if (num_sites < 2) SETERRQ1(mpi_comm, 1, "There must be at least two total sites. Got %lld.", LLD(num_sites));
        if (num_sites % 2) SETERRQ1(mpi_comm, 1, "Total number of sites must be even. Got %lld.", LLD(num_sites));

        /* EXTENSION, off by default: start every sweep step's eigen-solve from the transformed ground state of the previous step
           (csrc/predict.cpp) instead of the random vector the reference uses (:1484-1500) */
        o.GetBool("-wavefunction_prediction", &do_prediction, NULL);
        o.GetBool("-verbose", &verbose, NULL); if (o.Has("-verbose") && o.kv["-verbose"].empty()) verbose = PETSC_TRUE;
        o.GetBool("-no_symm", &no_symm, NULL);
        o.GetBool("-do_shell", &do_shell, NULL);
        o.GetBool("-dry_run", &dry_run, NULL); if (o.Has("-dry_run") && o.kv["-dry_run"].empty()) dry_run = PETSC_TRUE;
        o.GetReal("-qn_sector", &qn_sector, NULL);
        /* the SLEPc knobs of the "H_" prefixed EPS (:1494) */
        o.GetReal("-H_eps_tol", &eps_opts.tol, NULL);
        { PetscInt v = eps_opts.ncv; o.GetInt("-H_eps_ncv", &v, NULL); eps_opts.ncv = v; }
        { PetscInt v = eps_opts.max_it; o.GetInt("-H_eps_max_it", &v, NULL); eps_opts.max_it = v; }

        o.GetString("-scratch_dir", scratch_dir, &set);
        if (!set) { scratch_dir = "./scratch_dir/"; }
        if (scratch_dir.back() != '/') scratch_dir += '/';
        /* Blocks stay in HBM during a run; with an explicit -scratch_dir (or -save_blocks 1) every completed warm-up / sweep is
           checkpointed to Sweep_%09d/Sys_%09d/ in the reference's on-disk format so that -restart_dir can pick it up. */
        do_save_blocks = set;
        o.GetBool("-save_blocks", &do_save_blocks, NULL);
        { PetscInt v = io_int_bytes; o.GetInt("-petsc_int_bytes", &v, NULL); io_int_bytes = (int)v; }
        if (io_int_bytes != 4 && io_int_bytes != 8) SETERRQ(mpi_comm, 1, "-petsc_int_bytes must be 4 or 8");
        std::string data_dir;
        o.GetString("-data_dir", data_dir, &set);
        if (!set) data_dir = "./data_dir/";
        if (data_dir.back() != '/') data_dir += '/';
        ierr = Makedir(data_dir); CHKERRQ(ierr);

        fp_step = fopen((data_dir + "DMRGSteps.json").c_str(), "w");
        fp_timings = fopen((data_dir + "Timings.json").c_str(), "w");
        fp_entanglement = fopen((data_dir + "EntanglementSpectra.json").c_str(), "w");
        fp_data = fopen((data_dir + "DMRGRun.json").c_str(), "w");
        fp_corr = fopen((data_dir + "Correlations.json").c_str(), "w");
        if (!fp_step || !fp_timings || !fp_entanglement || !fp_data || !fp_corr) SETERRQ1(mpi_comm, 1, "cannot open output files in %s", data_dir.c_str());
        PetscBool do_corr_matrix = PETSC_FALSE, do_dimer_matrix = PETSC_FALSE, do_spectral = PETSC_FALSE, do_dyncorr = PETSC_FALSE;
        /* EXTENSION, off by default: the full two-point spin correlation matrix and the structure factor at every measurement
           step, in CorrelationMatrix.json; computed and written by rank 0 only */
        o.GetBool("-do_correlation_matrix", &do_corr_matrix, NULL);
        /* EXTENSION, off by default: the dimer (bond–bond) correlation matrix of the nearest-neighbour bonds and the dimer
           structure factors at every measurement step, in DimerMatrix.json; computed and written by rank 0 only */
        o.GetBool("-do_dimer_matrix", &do_dimer_matrix, NULL);
        /* EXTENSION, off by default: the dynamical structure factor S(q, ω) by the continued-fraction method at every measurement
           step, in SpectralFunction.json; computed and written by rank 0 of a single-GPU run */
        o.GetBool("-do_spectral_function", &do_spectral, NULL);
        o.GetInt("-spectral_nsteps", &spectral_nsteps, NULL);
        if (spectral_nsteps < 1) SETERRQ1(mpi_comm, 1, "-spectral_nsteps must be at least 1. Got %lld.", LLD(spectral_nsteps));
        if (o.Has("-spectral_ops")) {
            const std::vector<std::string> items = ListItems(o, "-spectral_ops");
            spectral_ops = {false, false, false};
            for (const std::string& item : items) {
                size_t k = 0;
                while (k < 3 && item != spectral_kinds[k].name) ++k;
                if (k == 3) SETERRQ1(mpi_comm, PETSC_ERR_ARG_WRONG, "-spectral_ops: unknown item '%s' (the items are zz, pm and mp).", item.c_str());
                spectral_ops[k] = true;
            }
            if (items.empty()) SETERRQ(mpi_comm, PETSC_ERR_ARG_WRONG, "-spectral_ops: the list is empty (the items are zz, pm and mp).");
        }
        /* EXTENSION, off by default: the real-space dynamical correlation matrix <O_s psi| f(H) |O_c psi> from single-site sources c
           at every measurement step, in DynamicalCorrelations.json (-spectral_nsteps, -spectral_ops); rank 0 of a single-GPU run */
        o.GetBool("-do_dynamical_correlations", &do_dyncorr, NULL);
        if (o.Has("-dynamical_sources")) {
            std::set<PetscInt> seen;
            for (const std::string& item : ListItems(o, "-dynamical_sources")) {
                size_t end = 0;
                long long v = -1;
                try { v = std::stoll(item, &end); } catch (...) { end = 0; }
                if (end != item.size() || v < 0 || v >= (long long)num_sites)
                    SETERRQ2(mpi_comm, PETSC_ERR_ARG_WRONG, "-dynamical_sources: '%s' is not a site index in [0, %lld).", item.c_str(), LLD(num_sites));
                if (!seen.insert((PetscInt)v).second) SETERRQ1(mpi_comm, PETSC_ERR_ARG_WRONG, "-dynamical_sources: site %lld is listed twice.", v);
                dyncorr_sources.push_back((PetscInt)v);
            }
            if (dyncorr_sources.empty()) SETERRQ(mpi_comm, PETSC_ERR_ARG_WRONG, "-dynamical_sources: the list is empty.");
        }
        {
            int rank = 0, world = 1;
            dmrgx_ctx_rank(DmrgxContext(), &rank, &world);
            /* the recurrence applies H on one GPU; the sharded apply is collective and a rank-0-only pass cannot use it */
            if (world > 1 && do_spectral) SETERRQ1(mpi_comm, PETSC_ERR_SUP, "-do_spectral_function runs on one GPU only (this run has %d ranks).", world);
            if (world > 1 && do_dyncorr)
                SETERRQ1(mpi_comm, PETSC_ERR_SUP, "-do_dynamical_correlations runs on one GPU only (this run has %d ranks).", world);
            if (rank != 0) do_corr_matrix = do_dimer_matrix = do_spectral = do_dyncorr = PETSC_FALSE;
        }
        if (do_corr_matrix) { ierr = corrmat.Open(data_dir, "CorrelationMatrix.json"); CHKERRQ(ierr); }
        if (do_dimer_matrix) { ierr = dimer.Open(data_dir, "DimerMatrix.json"); CHKERRQ(ierr); }
        if (do_spectral) { ierr = spectral.Open(data_dir, "SpectralFunction.json"); CHKERRQ(ierr); }
        if (do_dyncorr) { ierr = dyncorr.Open(data_dir, "DynamicalCorrelations.json"); CHKERRQ(ierr); }
        SaveStepHeaders(); fprintf(fp_step, "[\n");
        SaveTimingsHeaders(); fprintf(fp_timings, "[\n");
        fprintf(fp_entanglement, "[\n");
        fprintf(fp_data, "{\n"); Ham.SaveOut(fp_data); fprintf(fp_data, ",\n"); fprintf(fp_data, "  \"QNSector\": %g", qn_sector); fflush(fp_data);

        printf("=========================================\n"
               "DENSITY MATRIX RENORMALIZATION GROUP\n"
               "-----------------------------------------\n");
        Ham.PrintOut();
        printf("-----------------------------------------\n"
               "DIRECTORIES\n  Scratch: %s (blocks stay in HBM)\n  Data:    %s\n"
               "=========================================\n", scratch_dir.c_str(), data_dir.c_str());

        /* warm-up / sweep modes (:455-582) */
        PetscBool opt_mstates, opt_mwarmup, opt_nsweeps, opt_msweeps, opt_maxnsweeps;
        PetscInt mstates = 0;
        o.GetInt("-mstates", &mstates, &opt_mstates);
        o.GetInt("-mwarmup", &mwarmup, &opt_mwarmup);
        o.GetInt("-nsweeps", &nsweeps, &opt_nsweeps);
        o.GetIntArray("-msweeps", msweeps, &opt_msweeps);
        o.GetIntArray("-maxnsweeps", maxnsweeps, &opt_maxnsweeps);
        if (opt_mstates && !opt_mwarmup) mwarmup = mstates;
        if (opt_nsweeps && opt_msweeps) SETERRQ(mpi_comm, 1, "-msweeps and -nsweeps cannot both be specified at the same time.");
        if (opt_maxnsweeps && maxnsweeps.size() != msweeps.size())
            SETERRQ2(mpi_comm, 1, "-msweeps and -maxnsweeps must have the same number of items. Got %lld and %lld, respectively.",
                     LLD(msweeps.size()), LLD(maxnsweeps.size()));
        if (opt_nsweeps && !opt_msweeps) sweep_mode = SWEEP_MODE_NSWEEPS;
        else if (opt_msweeps && !opt_nsweeps) sweep_mode = opt_maxnsweeps ? SWEEP_MODE_TOLERANCE_TEST : SWEEP_MODE_MSWEEPS;
        else sweep_mode = SWEEP_MODE_NULL;

        std::cout << "WARMUP\n  NumStates to keep:           " << mwarmup << "\n";
        std::cout << "SWEEP\n  Sweep mode:                  " << SweepModeToString(sweep_mode) << std::endl;
        if (sweep_mode == SWEEP_MODE_NSWEEPS) std::cout << "  Number of sweeps:            " << nsweeps << std::endl;
        else if (sweep_mode == SWEEP_MODE_MSWEEPS) {
            std::cout << "  NumStates to keep:          ";
            for (const PetscInt& m : msweeps) std::cout << " " << m;
            std::cout << std::endl;
        } else if (sweep_mode == SWEEP_MODE_TOLERANCE_TEST) {
            std::cout << "  NumStates to keep, maxiter: ";
            for (size_t i = 0; i < msweeps.size(); ++i) std::cout << " (" << msweeps[i] << "," << maxnsweeps[i] << ")";
            std::cout << std::endl;
        }
        PrintLines();
        LoopType = WarmupStep;
        init = PETSC_TRUE;
        return 0;
    }

    /** :590-624 */
    PetscErrorCode Destroy() {
        if (!init) return 0;
        ClearPendingWaves();
        sys_bt.clear();
        SingleSite.Destroy();
        for (Block& blk : sys_blocks) blk.Destroy();
        fprintf(fp_step, "\n  ]\n}\n"); fclose(fp_step);
        fprintf(fp_timings, "\n  ]\n}\n"); fclose(fp_timings);
        fprintf(fp_entanglement, "\n]\n"); fclose(fp_entanglement);
        SaveLoopsData();
        fprintf(fp_data, "\n}\n"); fclose(fp_data);
        if (corr_headers_printed) fprintf(fp_corr, "\n  ]\n}\n");
        fclose(fp_corr);
        for (RecordFile* r : {&corrmat, &dimer, &spectral, &dyncorr}) r->Close();
        init = PETSC_FALSE;
        return 0;
    }

    /** :627-683 — site numbering of the superblock; environment sites are reflected */
    PetscErrorCode SetUpCorrelation(const std::vector<Op>& OpList, const std::string& name, const std::string& desc) {
        if (!init) SETERRQ(mpi_comm, 1, "DMRGBlockContainer object not initialized. Call Initialize() first.");
        if (LoopType == SweepStep) SETERRQ(mpi_comm, 1, "Setup correlation functions should be called before starting the sweeps.");
        Correlator m;
        m.idx = (PetscInt)measurements.size(); m.name = name; m.desc1 = desc;
        m.desc2 += "< ";
        for (const Op& op : OpList) m.desc2 += OpToStr(op.OpType) + "_{" + std::to_string(op.idx) + "} ";
        m.desc2 += ">";
        for (const Op& op : OpList) {
            if (0 <= op.idx && op.idx < num_sites / 2) m.SysOps.push_back(op);
            else if (num_sites / 2 <= op.idx && op.idx < num_sites) m.EnvOps.push_back({op.OpType, num_sites - 1 - op.idx});
            else SETERRQ2(mpi_comm, 1, "Operator index must be in the range [0,%lld). Got %lld.", LLD(num_sites), LLD(op.idx));
        }
        if (m.SysOps.empty()) { m.SysOps = m.EnvOps; m.EnvOps.clear(); }
        m.desc3 += "< ( ";
        for (const Op& op : m.SysOps) m.desc3 += OpToStr(op.OpType) + "_{" + std::to_string(op.idx) + "} ";
        if (m.SysOps.empty()) m.desc3 += "1 ";
        m.desc3 += ") ⊗ ( ";
        for (const Op& op : m.EnvOps) m.desc3 += OpToStr(op.OpType) + "_{" + std::to_string(op.idx) + "} ";
        if (m.EnvOps.empty()) m.desc3 += "1 ";
        m.desc3 += ") >";
        measurements.push_back(m);
        return 0;
    }

    /** :687-861 */
    PetscErrorCode Warmup() {
        if (!init) SETERRQ(mpi_comm, 1, "DMRGBlockContainer object not initialized. Call Initialize() first.");
        if (dry_run) return 0;
        if (mwarmup == 0 && !restart) { std::cout << "WARNING: Nothing left to do since mwarmup is zero." << std::endl; return 0; }
        PetscErrorCode ierr;
        t0abs = Now();
        if (restart) { /* the warm-up is replaced by loading the blocks of the previous run (:736-757) */
            std::cout << "Loading blocks from file..." << std::endl;
            if (num_sys_blocks != num_sites - 1) SETERRQ(mpi_comm, 1, "Sweep.dat does not belong to this lattice (num_sys_blocks).");
            sys_blocks.resize((size_t)num_sys_blocks);
            sys_bt.assign((size_t)num_sys_blocks, nullptr); sys_bt_src.assign((size_t)num_sys_blocks, -2);
            for (PetscInt iblock = 0; iblock < sys_ninit; ++iblock) {
                const std::string path_read = restart_dir + BlockDir("Sys", iblock);
                std::cout << "  Reading Block " << iblock << " from: " << path_read << std::endl;
                ierr = BlockIO::Load(sys_blocks[(size_t)iblock], path_read); CHKERRQ(ierr);
            }
            PrintLines();
            warmed_up = PETSC_TRUE;
            return 0;
        }
        if (warmed_up) SETERRQ(mpi_comm, 1, "Warmup has already been called, and it can only be called once.");
        printf("WARMUP\n");
        num_sys_blocks = num_sites - 1;
        sys_blocks.resize((size_t)num_sys_blocks);
        sys_bt.assign((size_t)num_sys_blocks, nullptr); sys_bt_src.assign((size_t)num_sys_blocks, -2);
        for (Block& b : sys_blocks) { ierr = b.Initialize(mpi_comm); CHKERRQ(ierr); }
        ierr = sys_blocks[(size_t)sys_ninit++].Initialize(mpi_comm, 1, PETSC_DEFAULT); CHKERRQ(ierr);
        if (AddSite.NumSites() != 1) SETERRQ1(mpi_comm, 1, "Routine assumes an additional site of 1. Got %lld.", LLD(AddSite.NumSites()));
        PetscInt nsites_cluster = Ham.NumEnvSites();
        if (nsites_cluster % 2) nsites_cluster *= 2;
        printf(" Preparing initial blocks.\n");
        while (sys_ninit < nsites_cluster) { /* exact blocks up to one cluster (:786-790) */
            const PetscInt NumSitesTotal = sys_blocks[(size_t)sys_ninit - 1].NumSites() + AddSite.NumSites();
            ierr = KronEye_Explicit(sys_blocks[(size_t)sys_ninit - 1], AddSite, Ham.H(NumSitesTotal), sys_blocks[(size_t)sys_ninit]); CHKERRQ(ierr);
            ++sys_ninit;
        }
        if (sys_ninit >= num_sites / 2)
            SETERRQ(mpi_comm, 1, "No DMRG Steps were performed since all site operators were created exactly.  Please change the system dimensions.");
        LoopType = WarmupStep;
        StepIdx = 0;
        while (sys_ninit < num_sites / 2) { /* :809-840 */
            PetscInt full_cluster = (((sys_ninit + 2) / nsites_cluster) + 1) * nsites_cluster;
            PetscInt env_numsites = full_cluster - sys_ninit - 2;
            const PetscInt env_add = ((sys_ninit - env_numsites) / nsites_cluster) * nsites_cluster;
            env_numsites += env_add;
            full_cluster += env_add;
            if (env_numsites < 1 || env_numsites > sys_ninit) SETERRQ1(mpi_comm, 1, "Incorrect number of sites. Got %lld.", LLD(env_numsites));
            if (verbose) PrintLines();
            printf(" %s  %lld/%lld/%lld\n", "WARMUP", LLD(LoopIdx), LLD(StepIdx), LLD(GlobIdx));
            PrintBlocks(sys_ninit, env_numsites);
            ierr = SingleDMRGStep(sys_blocks[(size_t)sys_ninit - 1], sys_blocks[(size_t)env_numsites - 1], mwarmup, sys_blocks[(size_t)sys_ninit],
                                  sys_blocks[(size_t)env_numsites], PetscBool(sys_ninit + 1 == num_sites / 2)); CHKERRQ(ierr);
            ++sys_ninit;
        }
        if (sys_ninit != num_sites / 2) SETERRQ2(mpi_comm, 1, "Expected sys_ninit = num_sites/2 = %lld. Got %lld.", LLD(num_sites / 2), LLD(sys_ninit));
        warmed_up = PETSC_TRUE;
        ierr = SaveSweepsData(); CHKERRQ(ierr);
        PrintLines();
        ++LoopIdx;
        return 0;
    }

    /** :864-993 */
    PetscErrorCode Sweeps() {
        if (dry_run || (mwarmup == 0 && !restart)) return 0;
        PetscErrorCode ierr;
        if (sweep_mode == SWEEP_MODE_NSWEEPS) {
            for (msweep_idx = 0; msweep_idx < nsweeps; ++msweep_idx) { ierr = SingleSweep(mwarmup); CHKERRQ(ierr); }
        } else if (sweep_mode == SWEEP_MODE_MSWEEPS) {
            for (msweep_idx = 0; msweep_idx < (PetscInt)msweeps.size(); ++msweep_idx) { ierr = SingleSweep(msweeps[(size_t)msweep_idx]); CHKERRQ(ierr); }
        } else if (sweep_mode == SWEEP_MODE_TOLERANCE_TEST) {
            for (msweep_idx = 0; msweep_idx < (PetscInt)msweeps.size(); ++msweep_idx) {
                const PetscInt mstates = msweeps[(size_t)msweep_idx], max_iter = maxnsweeps[(size_t)msweep_idx];
                PetscInt iter = 0;
                if (max_iter == 0) continue;
                bool cont;
                do { /* continue while |dE| > max truncation error and iter < max_iter (:945-953) */
                    const PetscScalar prev_gse = gse;
                    ierr = SingleSweep(mstates); CHKERRQ(ierr);
                    const PetscReal diff_gse = std::fabs(gse - prev_gse);
                    PetscReal max_trn = *std::max_element(trunc_err.begin(), trunc_err.end());
                    max_trn = std::max(max_trn, 0.0);
                    iter++;
                    cont = (iter < max_iter) && (diff_gse > max_trn);
                    std::cout << "SWEEP_MODE_TOLERANCE_TEST\n"
                              << "  Iterations / Max Iterations:       " << iter << "/" << max_iter << "\n"
                              << "  Difference in ground state energy: " << diff_gse << "\n"
                              << "  Largest truncation error:          " << max_trn << "\n"
                              << "  " << (cont ? "CONTINUE" : "BREAK") << std::endl;
                    PrintLines();
                } while (cont);
            }
        }
        return 0;
    }

    /** :996-1088 — centre to right, then (reflection symmetry) right-most block back to the midpoint */
    PetscErrorCode SingleSweep(const PetscInt& MStates, const PetscInt& MinBlock = PETSC_DEFAULT) {
        if (!init) SETERRQ(mpi_comm, 1, "DMRGBlockContainer object not initialized. Call Initialize() first.");
        PetscErrorCode ierr;
        if (!warmed_up) SETERRQ(mpi_comm, 1, "Warmup must be called first before performing sweeps.");
        printf("SWEEP MStates=%lld\n", LLD(MStates));
        const double tsweep0 = Now();
        trunc_err.clear();
        const PetscInt min_block = MinBlock == PETSC_DEFAULT ? 1 : MinBlock;
        if (min_block < 1) SETERRQ1(mpi_comm, 1, "MinBlock must at least be 1. Got %lld.", LLD(min_block));
        LoopType = SweepStep;
        StepIdx = 0;
        for (PetscInt iblock = num_sites / 2; iblock < num_sites - min_block - 2; ++iblock) {
            const PetscInt insys = iblock - 1, inenv = num_sites - iblock - 3;
            const PetscInt outsys = iblock, outenv = num_sites - iblock - 2;
            if (verbose) PrintLines();
            printf(" %s  %lld/%lld/%lld\n", "SWEEP", LLD(LoopIdx), LLD(StepIdx), LLD(GlobIdx));
            PrintBlocks(insys + 1, inenv + 1);
            ierr = SingleDMRGStep(sys_blocks[(size_t)insys], sys_blocks[(size_t)inenv], MStates, sys_blocks[(size_t)outsys], sys_blocks[(size_t)outenv]); CHKERRQ(ierr);
        }
        for (PetscInt iblock = min_block; iblock < num_sites / 2; ++iblock) {
            const PetscInt insys = num_sites - iblock - 3, inenv = iblock - 1;
            const PetscInt outsys = num_sites - iblock - 2, outenv = iblock;
            if (verbose) PrintLines();
            printf(" %s  %lld/%lld/%lld\n", "SWEEP", LLD(LoopIdx), LLD(StepIdx), LLD(GlobIdx));
            PrintBlocks(insys + 1, inenv + 1);
            ierr = SingleDMRGStep(sys_blocks[(size_t)insys], sys_blocks[(size_t)inenv], MStates, sys_blocks[(size_t)outsys], sys_blocks[(size_t)outenv],
                                  PetscBool(outsys == outenv)); CHKERRQ(ierr);
        }
        sweeps_mstates.push_back(MStates);
        sweeps_seconds.push_back(Now() - tsweep0);
        printf("  Sweep time: %.6f s (%lld steps)\n", sweeps_seconds.back(), LLD(StepIdx));
        ierr = SaveSweepsData(); CHKERRQ(ierr);
        ++LoopIdx;
        PrintLines();
        return 0;
    }

    const Block& SysBlock(const PetscInt& BlockIdx) const {
        if (BlockIdx >= sys_ninit) throw std::runtime_error("Attempted to access uninitialized system block.");
        return sys_blocks[(size_t)BlockIdx];
    }
    PetscInt NumSites() const { return num_sites; }
    PetscBool Verbose() const { return verbose; }
    const Hamiltonian& HamiltonianRef() const { return Ham; }
    PetscScalar GroundStateEnergy() const { return gse; }
    const std::vector<double>& SweepSeconds() const { return sweeps_seconds; }

private:
    typedef enum { SWEEP_MODE_NULL, SWEEP_MODE_NSWEEPS, SWEEP_MODE_MSWEEPS, SWEEP_MODE_TOLERANCE_TEST } SweepMode_t;
    typedef enum { WarmupStep = 0, SweepStep = 1, NullStep = 2 } Step_t;
    /** An extension's output file: a JSON array with one record per measurement step, each record opening with GlobIdx and
        LoopIdx.  The record count places the commas between records. */
    struct RecordFile {
        FILE* f = NULL;
        long long records = 0;
        explicit operator bool() const { return f != NULL; }
        PetscErrorCode Open(const std::string& data_dir, const char* name) {
            f = fopen((data_dir + name).c_str(), "w");
            if (!f) SETERRQ2(PETSC_COMM_SELF, 1, "cannot open %s%s", data_dir.c_str(), name);
            fprintf(f, "[\n"); fflush(f);
            return 0;
        }
        FILE* BeginRecord(PetscInt GlobIdx, PetscInt LoopIdx) {
            fprintf(f, "%s  {\n    \"GlobIdx\": %lld,\n    \"LoopIdx\": %lld", records ? ",\n" : "", LLD(GlobIdx), LLD(LoopIdx));
            return f;
        }
        void EndRecord() { fprintf(f, "\n  }"); fflush(f); ++records; }
        void Close() { if (f) { fprintf(f, "\n]\n"); fclose(f); f = NULL; } }
    };
    /** The lattice coordinates (x[s], y[s]) of points s */
    struct Coords { std::vector<PetscInt> x, y; };
    /** The recurrences of -do_spectral_function and -do_dynamical_correlations, in the order of -spectral_ops' flags */
    struct SpectralKind { const char* name; int op; };
    static constexpr SpectralKind spectral_kinds[3] = {{"zz", DMRGX_OP_SZ}, {"pm", DMRGX_OP_SM}, {"mp", DMRGX_OP_SP}};
    /** The items of a list option, separated by commas or blanks; empty items are dropped */
    static std::vector<std::string> ListItems(PetscOptions& o, const char* key) {
        std::string list;
        o.GetString(key, list, NULL);
        for (char& c : list) if (c == ',') c = ' ';
        std::istringstream iss(list);
        std::vector<std::string> items;
        for (std::string item; iss >> item;) items.push_back(item);
        return items;
    }
    static const char* SweepModeToString(SweepMode_t m) {
        switch (m) {
            case SWEEP_MODE_NSWEEPS: return "SWEEP_MODE_NSWEEPS";
            case SWEEP_MODE_MSWEEPS: return "SWEEP_MODE_MSWEEPS";
            case SWEEP_MODE_TOLERANCE_TEST: return "SWEEP_MODE_TOLERANCE_TEST";
            default: return "SWEEP_MODE_NULL";
        }
    }
    /** :96-139 */
    struct StepData {
        PetscInt NumSites_Sys, NumSites_Env, NumSites_SysEnl, NumSites_EnvEnl, NumStates_Sys, NumStates_Env, NumStates_SysEnl, NumStates_EnvEnl,
            NumStates_SysRot, NumStates_EnvRot, NumStates_H;
        PetscScalar GSEnergy;
        PetscReal TruncErr_Sys, TruncErr_Env;
    };
    struct TimingsData { double tEnlr, tKron, tDiag, tRdms, tRotb, Total; };

    static double Now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
    /* phase boundaries are wall-clock like PetscTime, taken after the device went idle */
    static double Tick() { dmrgx_ctx_sync(DmrgxContext()); return Now(); }
    static void PrintLines() { printf("-----------------------------------------\n"); }
    void PrintBlocks(const PetscInt& nsys, const PetscInt& nenv) const {
        printf("  [");
        for (PetscInt i = 0; i < nsys; ++i) printf("=");
        printf("**");
        for (PetscInt i = 0; i < nenv; ++i) printf("-");
        printf("]\n");
    }

    /** :1304-1653 */
    PetscErrorCode SingleDMRGStep(Block& SysBlock, Block& EnvBlock, const PetscInt& MStates, Block& SysBlockOut, Block& EnvBlockOut,
                                  PetscBool do_measurements = PETSC_FALSE) {
        PetscErrorCode ierr;
        TimingsData timings_data;
        const double t0 = t0abs;
        StepData step_data;
        step_data.NumSites_Sys = SysBlock.NumSites();
        step_data.NumSites_Env = EnvBlock.NumSites();
        step_data.NumStates_Sys = SysBlock.NumStates();
        step_data.NumStates_Env = EnvBlock.NumStates();
        const PetscBool flg = PetscBool(&SysBlock == &EnvBlock);

        /* add one site to each block */
        Block SysBlockEnl, EnvBlockEnl;
        ierr = KronEye_Explicit(SysBlock, AddSite, Ham.H(SysBlock.NumSites() + AddSite.NumSites()), SysBlockEnl); CHKERRQ(ierr);
        if (!flg) { ierr = KronEye_Explicit(EnvBlock, AddSite, Ham.H(EnvBlock.NumSites() + AddSite.NumSites()), EnvBlockEnl); CHKERRQ(ierr); }
        else EnvBlockEnl = SysBlockEnl;
        const double tenlr = Tick();
        timings_data.tEnlr = tenlr - t0;
        if (verbose) printf("* Add One Site:          %12.6f s\n", timings_data.tEnlr);
        step_data.NumSites_SysEnl = SysBlockEnl.NumSites();
        step_data.NumSites_EnvEnl = EnvBlockEnl.NumSites();
        step_data.NumStates_SysEnl = SysBlockEnl.NumStates();
        step_data.NumStates_EnvEnl = EnvBlockEnl.NumStates();

        /* superblock Hamiltonian */
        const PetscInt NumSitesTotal = SysBlockEnl.NumSites() + EnvBlockEnl.NumSites();
        const std::vector<Hamiltonians::Term> Terms = Ham.H(NumSitesTotal);
        std::vector<PetscReal> QNSectors = {qn_sector};
        if (no_symm) QNSectors = {};
        KronBlocks_t KronBlocks(SysBlockEnl, EnvBlockEnl, QNSectors, NULL, GlobIdx);
        step_data.NumStates_H = KronBlocks.NumStates();
        ShellMat H;
        ierr = KronBlocks.KronSumSetRedistribute(PETSC_TRUE); CHKERRQ(ierr);
        ierr = KronBlocks.KronSumSetToleranceFromOptions(); CHKERRQ(ierr);
        ierr = KronBlocks.KronSumSetShellMatrix(do_shell); CHKERRQ(ierr);
        ierr = KronBlocks.KronSumConstruct(Terms, H); CHKERRQ(ierr);
        if (!H) SETERRQ(mpi_comm, 1, "H is null.");
        const double tkron = Tick();
        timings_data.tKron = tkron - tenlr;
        if (verbose) printf("* Build Superblock H:    %12.6f s\n", timings_data.tKron);

        /* ground state (EPS_HEP, EPS_SMALLEST_REAL, nev = 1) */
        Vec gsv_r;
        ierr = MatCreateVecs(H, &gsv_r); CHKERRQ(ierr);
        PetscScalar gse_r = 0;
        dmrgx_eigs_stats eps_stats;
        eps_opts.seed = 20261018ULL + (unsigned long long)GlobIdx;
        /* -wavefunction_prediction: the previous step's ground state carried over to this superblock, when the blocks chain up */
        Vec guess;
        PetscBool predicted = PETSC_FALSE;
        const long long idx_sys = BlockIndex(SysBlock), idx_env = BlockIndex(EnvBlock);
        if (do_prediction && (pending.wL || pending.wR)) {
            int ok = 0;
            ierr = MatCreateVecs(H, &guess); CHKERRQ(ierr);
            if (pending.wL && pending.out_sys == SysBlock.Serial() && pending.xe_left && pending.xe_left_src == EnvBlock.Serial()) {
                DMRGX_CALL(dmrgx_wave_apply(pending.wL, pending.xe_left->h, AddSite.Handle(), KronBlocks.Handle(), guess.d, &ok));
            } else if (pending.wR && pending.out_env == EnvBlock.Serial() && pending.xe_right && pending.xe_right_src == SysBlock.Serial()) {
                DMRGX_CALL(dmrgx_wave_apply(pending.wR, pending.xe_right->h, AddSite.Handle(), KronBlocks.Handle(), guess.d, &ok));
            }
            predicted = PetscBool(ok != 0);
            if (predicted) ++steps_predicted;
        }
        ClearPendingWaves();
        DMRGX_CALL(dmrgx_eigs_smallest_from(H.h, &eps_opts, predicted ? guess.d : NULL, &gse_r, gsv_r.d, &eps_stats));
        if (guess.d) { ierr = VecDestroy(&guess); CHKERRQ(ierr); }
        step_data.GSEnergy = gse_r;
        total_matvecs += eps_stats.nmatvec;
        double h_bytes = 0, h_flops = 0;
        { dmrgx_int hn, hnt, t1, t2; dmrgx_hshell_stats(H.h, &hn, &hnt, &h_bytes, &h_flops, &t1, &t2); }
        /* -do_spectral_function, -do_dynamical_correlations: the zz recurrence runs on this step's H, which then lives until the
           measurement */
        if (!(do_measurements && (spectral || dyncorr))) { ierr = MatDestroy_KronSumShell(&H); CHKERRQ(ierr); }
        const double tdiag = Tick();
        total_matvec_flops += h_flops * (double)eps_stats.nmatvec;
        timings_data.tDiag = tdiag - tkron;
        if (verbose) printf("* Solve Ground State:    %12.6f s   (%lld H*psi of %.2f GFLOP, %.1f TFLOP/s incl. orthogonalisation, residual %.3g%s)\n",
                            timings_data.tDiag, LLD(eps_stats.nmatvec), h_flops * 1e-9, h_flops * (double)eps_stats.nmatvec / timings_data.tDiag * 1e-12,
                            eps_stats.resid, eps_stats.converged ? "" : ", NOT converged");
        if (no_symm) SETERRQ(mpi_comm, PETSC_ERR_SUP, "Unsupported option: no_symm.");

        /* reduced density matrices and the rotation */
        std::shared_ptr<BasisTransformation> pBT_L = std::make_shared<BasisTransformation>(), pBT_R = std::make_shared<BasisTransformation>();
        BasisTransformation &BT_L = *pBT_L, &BT_R = *pBT_R;
        DMRGX_CALL(dmrgx_truncate(KronBlocks.Handle(), gsv_r.d, MStates, &BT_L.h, &BT_R.h));
        ierr = BT_L.Load(); CHKERRQ(ierr);
        ierr = BT_R.Load(); CHKERRQ(ierr);
        ierr = SaveEntanglementSpectra(BT_L, SysBlockEnl.Magnetization.List(), BT_R, EnvBlockEnl.Magnetization.List()); CHKERRQ(ierr);
        ierr = CalculateCorrelations_BlockDiag(KronBlocks, gsv_r, do_measurements); CHKERRQ(ierr);
        const Coords r = do_measurements ? SiteCoords(NumSitesTotal) : Coords();
        if (do_measurements && corrmat) { ierr = CalculateCorrelationMatrix(KronBlocks, gsv_r, r); CHKERRQ(ierr); }
        if (do_measurements && dimer) { ierr = CalculateDimerMatrix(KronBlocks, gsv_r); CHKERRQ(ierr); }
        if (do_measurements && spectral) { ierr = CalculateSpectralFunction(KronBlocks, H, gsv_r, gse_r, r, Terms, SysBlockEnl, EnvBlockEnl); CHKERRQ(ierr); }
        if (do_measurements && dyncorr) { ierr = CalculateDynamicalCorrelations(KronBlocks, H, gsv_r, gse_r, r, Terms, SysBlockEnl, EnvBlockEnl); CHKERRQ(ierr); }
        if (do_measurements && (spectral || dyncorr)) { ierr = MatDestroy_KronSumShell(&H); CHKERRQ(ierr); }
        if (do_prediction) {
            /* both candidates: which block grows in the next step is the caller's business (the left one in the first half of a sweep,
               the right one in the second, :996-1088); the transformations that created this step's input blocks are captured now,
               before this step's outputs replace entries of sys_bt */
            DMRGX_CALL(dmrgx_wave_create(KronBlocks.Handle(), gsv_r.d, BT_L.h, 1, &pending.wL));
            if (!flg) DMRGX_CALL(dmrgx_wave_create(KronBlocks.Handle(), gsv_r.d, BT_R.h, 0, &pending.wR));
            if (idx_env >= 0) { pending.xe_left = sys_bt[(size_t)idx_env]; pending.xe_left_src = sys_bt_src[(size_t)idx_env]; }
            if (idx_sys >= 0) { pending.xe_right = sys_bt[(size_t)idx_sys]; pending.xe_right_src = sys_bt_src[(size_t)idx_sys]; }
        }
        const long long serial_sys_in = SysBlock.Serial(), serial_env_in = EnvBlock.Serial();
        ierr = VecDestroy(&gsv_r); CHKERRQ(ierr);
        const double trdms = Tick();
        timings_data.tRdms = trdms - tdiag;
        if (verbose) printf("* Eigendec. of RDMs:     %12.6f s\n", timings_data.tRdms);

        /* new blocks: outputs may alias the inputs (entries of sys_blocks), so rotate into fresh handles first */
        dmrgx_block newsys = nullptr, newenv = nullptr;
        DMRGX_CALL(dmrgx_rotate(SysBlockEnl.Handle(), BT_L.h, &newsys));
        if (!flg) DMRGX_CALL(dmrgx_rotate(EnvBlockEnl.Handle(), BT_R.h, &newenv));
        ierr = SysBlockOut.Adopt(newsys); CHKERRQ(ierr);
        if (!flg) { ierr = EnvBlockOut.Adopt(newenv); CHKERRQ(ierr); }
        if (do_prediction) {
            const long long osys = BlockIndex(SysBlockOut), oenv = BlockIndex(EnvBlockOut);
            if (osys >= 0) { sys_bt[(size_t)osys] = pBT_L; sys_bt_src[(size_t)osys] = serial_sys_in; }
            if (!flg && oenv >= 0) { sys_bt[(size_t)oenv] = pBT_R; sys_bt_src[(size_t)oenv] = serial_env_in; }
            pending.out_sys = SysBlockOut.Serial();
            pending.out_env = flg ? -1 : EnvBlockOut.Serial();
        }
        step_data.NumStates_SysRot = SysBlockOut.NumStates();
        step_data.NumStates_EnvRot = EnvBlockOut.NumStates();
        step_data.TruncErr_Sys = BT_L.TruncErr;
        step_data.TruncErr_Env = BT_R.TruncErr;
        const double trotb = Tick();
        timings_data.tRotb = trotb - trdms;
        if (verbose) printf("* Rotation of Operators: %12.6f s\n", timings_data.tRotb);
        timings_data.Total = trotb - t0;
        t0abs = Now();

        if (verbose) {
            printf("\n  Superblock:\n    NumStates:      %lld\n    NumSites:       %lld\n    QNSector:       %-10.10g\n    Energy:         %-10.10g\n"
                   "    Energy/site:    %-10.10g\n", LLD(KronBlocks.NumStates()), LLD(NumSitesTotal), qn_sector, gse_r, gse_r / PetscReal(NumSitesTotal));
            printf("  Sys Block Out\n    NumStates:      %lld\n    TrunError:      %g\n", LLD(BT_L.QN.NumStates()), BT_L.TruncErr);
            printf("  Env Block Out\n    NumStates:      %lld\n    TrunError:      %g\n\n", LLD(BT_R.QN.NumStates()), BT_R.TruncErr);
            printf("  Total Time:              %12.6f s\n", timings_data.Total);
        }
        gse = gse_r;
        trunc_err.push_back(BT_L.TruncErr);
        ierr = SaveStepData(step_data); CHKERRQ(ierr);
        ierr = SaveTimingsData(timings_data); CHKERRQ(ierr);
        ++GlobIdx;
        ++StepIdx;
        ++rows_written;
        return 0;
    }

    /** :2062-2337 — <psi| (prod SysOps) ⊗ (prod EnvOps) |psi> through KronConstruct + MatMult + VecDot.  Products of
        several operators on one block are built on the device by dmrgx_block_op_product. */
    PetscErrorCode CalculateCorrelations_BlockDiag(KronBlocks_t& KronBlocks, const Vec& gsv_r, const PetscBool flg = PETSC_TRUE) {
        if (!corr_headers_printed) {
            fprintf(fp_corr, "{\n  \"info\" :\n  [\n");
            for (size_t icorr = 0; icorr < measurements.size(); ++icorr) {
                if (icorr) fprintf(fp_corr, ",\n");
                const Correlator& c = measurements[icorr];
                fprintf(fp_corr, "    {\n      \"corrIdx\" : %lld,\n      \"name\"    : \"%s\",\n      \"desc1\"   : \"%s\",\n      \"desc2\"   : \"%s\",\n"
                                 "      \"desc3\"   : \"%s\"\n    }", LLD(c.idx), c.name.c_str(), c.desc1.c_str(), c.desc2.c_str(), c.desc3.c_str());
            }
            fprintf(fp_corr, "\n  ],\n  \"values\" :\n  [\n");
            fflush(fp_corr);
            corr_headers_printed = PETSC_TRUE;
        }
        if (!flg) return 0;
        std::vector<PetscScalar> CorrValues(measurements.size(), 0.0);
        for (size_t icorr = 0; icorr < measurements.size(); ++icorr) {
            const Correlator& c = measurements[icorr];
            std::vector<int> lops, rops; std::vector<dmrgx_int> lsites, rsites;
            for (const Op& op : c.SysOps) { lops.push_back((int)op.OpType); lsites.push_back(op.idx); }
            for (const Op& op : c.EnvOps) { rops.push_back((int)op.OpType); rsites.push_back(op.idx); }
            dmrgx_hshell h1 = nullptr;
            DMRGX_CALL(dmrgx_hshell_create_product(KronBlocks.Handle(), (dmrgx_int)lops.size(), lops.data(), lsites.data(), (dmrgx_int)rops.size(),
                                                   rops.data(), rsites.data(), &h1));
            PetscScalar v = 0;
            const int e = dmrgx_expect(h1, gsv_r.d, &v);
            dmrgx_hshell_destroy(h1);
            if (e) return e;
            CorrValues[icorr] = v;
        }
        if (corr_printed_first) fprintf(fp_corr, ",\n");
        corr_printed_first = PETSC_TRUE;
        fprintf(fp_corr, "    [");
        for (size_t icorr = 0; icorr < measurements.size(); ++icorr) fprintf(fp_corr, "%s %g", icorr ? "," : "", CorrValues[icorr]);
        fprintf(fp_corr, " ]");
        fflush(fp_corr);
        return 0;
    }

    /** `,\n    "name": [[...], ...]` — a rows×cols row-major matrix of a CorrelationMatrix.json / DimerMatrix.json record, %.17g */
    static void WriteJsonMatrix(FILE* f, const char* name, const std::vector<double>& m, size_t rows, size_t cols) {
        fprintf(f, ",\n    \"%s\": [", name);
        for (size_t i = 0; i < rows; ++i) {
            fprintf(f, "%s\n      [", i ? "," : "");
            for (size_t j = 0; j < cols; ++j) fprintf(f, "%s%.17g", j ? ", " : "", m[i * cols + j]);
            fprintf(f, "]");
        }
        fprintf(f, "\n    ]");
    }

    /** The lattice coordinates of the sites of an nsites-site superblock (superblock site s is lattice site s) */
    Coords SiteCoords(const PetscInt nsites) const {
        Coords r{std::vector<PetscInt>((size_t)nsites), std::vector<PetscInt>((size_t)nsites)};
        for (PetscInt s = 0; s < nsites; ++s) Ham.To2D(s, r.x[(size_t)s], r.y[(size_t)s]);
        return r;
    }
    /** `,\n    "sites": [[x, y], ...]` of a record */
    static void WriteSites(FILE* f, const Coords& r) {
        fprintf(f, ",\n    \"sites\": [");
        for (size_t s = 0; s < r.x.size(); ++s) fprintf(f, "%s[%lld, %lld]", s ? ", " : "", LLD(r.x[s]), LLD(r.y[s]));
        fprintf(f, "]");
    }
    /** The structure factor (1/N) Σ_ab cos(q·(r_a - r_b)) M_ab of the N points r and the N×N row-major M, for every
        q = (2π kx/Lx, 2π ky/Ly), as [kx][ky]; all zero when there is no point */
    std::vector<double> StructureFactor(const Coords& r, const std::vector<double>& M) const {
        const PetscInt Lx = Ham.Lx(), Ly = Ham.Ly();
        const size_t n = r.x.size();
        std::vector<double> sq((size_t)(Lx * Ly), 0.0);
        for (PetscInt kx = 0; kx < Lx && n > 0; ++kx)
            for (PetscInt ky = 0; ky < Ly; ++ky) {
                const double qx = 2.0 * M_PI * (double)kx / (double)Lx, qy = 2.0 * M_PI * (double)ky / (double)Ly;
                double s = 0;
                for (size_t a = 0; a < n; ++a)
                    for (size_t b = 0; b < n; ++b)
                        s += std::cos(qx * (double)(r.x[a] - r.x[b]) + qy * (double)(r.y[a] - r.y[b])) * M[a * n + b];
                sq[(size_t)(kx * Ly + ky)] = s / (double)n;
            }
        return sq;
    }
    /** `"alpha": [...], "beta": [...]` — the first `steps` coefficients of a recurrence */
    static void WriteAlphaBeta(FILE* f, const double* alpha, const double* beta, const dmrgx_int steps) {
        fprintf(f, "\"alpha\": [");
        for (dmrgx_int t = 0; t < steps; ++t) fprintf(f, "%s%.17g", t ? ", " : "", alpha[t]);
        fprintf(f, "], \"beta\": [");
        for (dmrgx_int t = 0; t < steps; ++t) fprintf(f, "%s%.17g", t ? ", " : "", beta[t]);
        fprintf(f, "]");
    }

    /** EXTENSION (-do_correlation_matrix): one record of CorrelationMatrix.json — every <S_i S_j> of the superblock from
        dmrgx_corr_matrix (superblock site s is lattice site s), and the static structure factor
            S(q) = (1/N) Σ_ij cos(q·(r_i - r_j)) <S_i·S_j>,   <S_i·S_j> = SzSz + (SpSm + SmSp)/2,   q = (2π kx/Lx, 2π ky/Ly),
        written as StructureFactor[kx][ky]. */
    PetscErrorCode CalculateCorrelationMatrix(KronBlocks_t& KronBlocks, const Vec& gsv_r, const Coords& r) {
        const size_t n = r.x.size();
        std::vector<double> szsz(n * n), spsm(n * n), smsp(n * n), sz(n);
        DMRGX_CALL(dmrgx_corr_matrix(KronBlocks.Handle(), gsv_r.d, szsz.data(), spsm.data(), smsp.data(), sz.data(), NULL));
        FILE* f = corrmat.BeginRecord(GlobIdx, LoopIdx);
        WriteSites(f, r);
        fprintf(f, ",\n    \"Sz\": [");
        for (size_t s = 0; s < n; ++s) fprintf(f, "%s%.17g", s ? ", " : "", sz[s]);
        fprintf(f, "]");
        WriteJsonMatrix(f, "SzSz", szsz, n, n);
        WriteJsonMatrix(f, "SpSm", spsm, n, n);
        WriteJsonMatrix(f, "SmSp", smsp, n, n);
        std::vector<double> ss(n * n);
        for (size_t k = 0; k < n * n; ++k) ss[k] = szsz[k] + 0.5 * (spsm[k] + smsp[k]);
        WriteJsonMatrix(f, "StructureFactor", StructureFactor(r, ss), (size_t)Ham.Lx(), (size_t)Ham.Ly());
        corrmat.EndRecord();
        return 0;
    }

    /** EXTENSION (-do_dimer_matrix): one record of DimerMatrix.json — the dimer correlations of the distinct nearest-neighbour
        bonds a = (i, j) of the lattice (Ham.NeighborPairs(), i < j; superblock site s is lattice site s) from dmrgx_dimer_matrix:
            Dimer[a] = <D_a>,  DimerDimer[a][b] = <D_a D_b>,  D_a = S_i·S_j,
        and per orientation α in {x, y} the dimer structure factor
            S_D^α(q) = (1/N_α) Σ_{a,b∈α} cos(q·(r_a - r_b)) (<D_a D_b> - <D_a><D_b>),   q = (2π kx/Lx, 2π ky/Ly),
        written as DimerStructureFactorX / Y [kx][ky] (all zero when the lattice has no bond of that orientation).  r_a is the
        bond's origin, the site from which the +x or +y step leads (for a wrap-around bond the one at x = Lx - 1 or y = Ly - 1). */
    PetscErrorCode CalculateDimerMatrix(KronBlocks_t& KronBlocks, const Vec& gsv_r) {
        const PetscInt Lx = Ham.Lx(), Ly = Ham.Ly();
        struct Bond { PetscInt i, j, xi, yi, xj, yj, ox, oy; char dir; };
        std::vector<Bond> bonds;
        { /* Ly = 2 with periodic y lists every vertical bond twice */
            std::set<std::pair<PetscInt, PetscInt>> seen;
            for (const std::vector<PetscInt>& p : Ham.NeighborPairs()) {
                if (!seen.insert({p[0], p[1]}).second) continue;
                Bond b;
                b.i = p[0]; b.j = p[1];
                Ham.To2D(b.i, b.xi, b.yi); Ham.To2D(b.j, b.xj, b.yj);
                b.dir = b.xi == b.xj ? 'y' : 'x';
                const PetscInt ui = b.dir == 'y' ? b.yi : b.xi, uj = b.dir == 'y' ? b.yj : b.xj;
                const bool from_i = ui + 1 == uj || (uj + 1 != ui && ui > uj); /* a +1 step, else the wrap-around from the last row */
                b.ox = from_i ? b.xi : b.xj; b.oy = from_i ? b.yi : b.yj;
                bonds.push_back(b);
            }
        }
        const size_t nb = bonds.size();
        if (nb == 0) SETERRQ(mpi_comm, 1, "-do_dimer_matrix: the lattice has no nearest-neighbour bond.");
        std::vector<dmrgx_int> si(nb), sj(nb);
        for (size_t a = 0; a < nb; ++a) { si[a] = bonds[a].i; sj[a] = bonds[a].j; }
        std::vector<double> dd(nb * nb), d(nb);
        DMRGX_CALL(dmrgx_dimer_matrix(KronBlocks.Handle(), gsv_r.d, (dmrgx_int)nb, si.data(), sj.data(), dd.data(), d.data(), NULL));
        FILE* f = dimer.BeginRecord(GlobIdx, LoopIdx);
        fprintf(f, ",\n    \"bonds\": [");
        for (size_t a = 0; a < nb; ++a) {
            const Bond& b = bonds[a];
            fprintf(f, "%s\n      {\"sites\": [%lld, %lld], \"coords\": [[%lld, %lld], [%lld, %lld]], \"orientation\": \"%c\", \"origin\": [%lld, %lld]}",
                    a ? "," : "", LLD(b.i), LLD(b.j), LLD(b.xi), LLD(b.yi), LLD(b.xj), LLD(b.yj), b.dir, LLD(b.ox), LLD(b.oy));
        }
        fprintf(f, "\n    ],\n    \"Dimer\": [");
        for (size_t a = 0; a < nb; ++a) fprintf(f, "%s%.17g", a ? ", " : "", d[a]);
        fprintf(f, "]");
        WriteJsonMatrix(f, "DimerDimer", dd, nb, nb);
        for (const char dir : {'x', 'y'}) {
            std::vector<size_t> in;
            Coords origins;
            for (size_t a = 0; a < nb; ++a)
                if (bonds[a].dir == dir) { in.push_back(a); origins.x.push_back(bonds[a].ox); origins.y.push_back(bonds[a].oy); }
            const size_t m = in.size();
            std::vector<double> conn(m * m);
            for (size_t a = 0; a < m; ++a)
                for (size_t b = 0; b < m; ++b) conn[a * m + b] = dd[in[a] * nb + in[b]] - d[in[a]] * d[in[b]];
            WriteJsonMatrix(f, dir == 'x' ? "DimerStructureFactorX" : "DimerStructureFactorY", StructureFactor(origins, conn), (size_t)Lx, (size_t)Ly);
        }
        dimer.EndRecord();
        return 0;
    }

    /** The target shell of the recurrences of op at this step, handed to `call` (which returns a dmrgx code): this step's H for
        Sz, else a shell on the sector qn + op built from the enlarged blocks and destroyed afterwards.  An empty shifted sector
        makes no call, so its outputs stay zero. */
    template <class F>
    PetscErrorCode WithSpectralTarget(const ShellMat& H, int op, const std::vector<Hamiltonians::Term>& Terms, Block& SysBlockEnl, Block& EnvBlockEnl,
                                      const char* what, F&& call) {
        if (op == DMRGX_OP_SZ) {
            const int e = call(H.h);
            if (e) fprintf(stderr, "[dmrgx] %s -> %d: %s\n", what, e, dmrgx_last_error());
            return e;
        }
        KronBlocks_t shifted(SysBlockEnl, EnvBlockEnl, {qn_sector + op}, NULL, GlobIdx);
        if (shifted.NumStates() == 0) return 0;
        ShellMat Hs;
        PetscErrorCode ierr = shifted.KronSumConstruct(Terms, Hs); CHKERRQ(ierr);
        const int e = call(Hs.h);
        if (e) fprintf(stderr, "[dmrgx] %s: %s\n", what, dmrgx_last_error());
        ierr = MatDestroy_KronSumShell(&Hs); CHKERRQ(ierr);
        return e;
    }

    /** EXTENSION (-do_spectral_function): one record of SpectralFunction.json — the continued-fraction coefficients of the
        dynamical structure factor from dmrgx_spectral_lanczos.  For every q = (2π kx/Lx, 2π ky/Ly) the start vectors are
            A_cos psi = Σ_s cos(q·r_s)/√N · O_s psi,   A_sin psi = Σ_s sin(q·r_s)/√N · O_s psi   (superblock site s is lattice site s),
        so that for a real psi and H  S(q, ω) = S_cos(ω) + S_sin(ω), with S_part(ω) = -Im G_part(ω + E0 + iη) / π and
        G = norm2 / (z - α_0 - β_1² / (z - α_1 - …)).  zz takes O = Sz under this step's H; pm = <S+ S-> takes O = S- under the H of
        the sector qn - 1 and mp = <S- S+> takes O = S+ under the H of the sector qn + 1, both built from the enlarged blocks.  An
        empty shifted sector gives zeros.  Written per operator as [kx][ky] -> {"cos": ..., "sin": ...}, each part holding norm2,
        steps (the recurrence length) and the first `steps` of alpha and beta (beta[0] = 0).  At equal time,
        Σ_parts (zz + (pm + mp)/2) norm2 = StructureFactor[kx][ky] of CorrelationMatrix.json. */
    PetscErrorCode CalculateSpectralFunction(KronBlocks_t& KronBlocks, const ShellMat& H, const Vec& gsv_r, const PetscScalar E0, const Coords& r,
                                             const std::vector<Hamiltonians::Term>& Terms, Block& SysBlockEnl, Block& EnvBlockEnl) {
        const PetscInt Lx = Ham.Lx(), Ly = Ham.Ly();
        const size_t n = r.x.size(), nq = (size_t)(Lx * Ly), nvec = 2 * nq, ns = (size_t)spectral_nsteps;
        std::vector<double> coef(nvec * n);
        for (PetscInt kx = 0; kx < Lx; ++kx)
            for (PetscInt ky = 0; ky < Ly; ++ky) {
                const double qx = 2.0 * M_PI * (double)kx / (double)Lx, qy = 2.0 * M_PI * (double)ky / (double)Ly;
                const size_t v = 2 * (size_t)(kx * Ly + ky);
                for (size_t s = 0; s < n; ++s) {
                    const double ph = qx * (double)r.x[s] + qy * (double)r.y[s];
                    coef[v * n + s] = std::cos(ph) / std::sqrt((double)n);
                    coef[(v + 1) * n + s] = std::sin(ph) / std::sqrt((double)n);
                }
            }
        FILE* f = spectral.BeginRecord(GlobIdx, LoopIdx);
        fprintf(f, ",\n    \"E0\": %.17g,\n    \"NSteps\": %lld", E0, LLD(spectral_nsteps));
        WriteSites(f, r);
        for (size_t k = 0; k < 3; ++k) {
            if (!spectral_ops[k]) continue;
            const SpectralKind& kind = spectral_kinds[k];
            std::vector<double> alpha(nvec * ns, 0.0), beta(nvec * ns, 0.0), norm2(nvec, 0.0);
            std::vector<dmrgx_int> steps(nvec, 0);
            PetscErrorCode ierr = WithSpectralTarget(H, kind.op, Terms, SysBlockEnl, EnvBlockEnl, "dmrgx_spectral_lanczos", [&](dmrgx_hshell t) {
                return dmrgx_spectral_lanczos(KronBlocks.Handle(), gsv_r.d, t, kind.op, (dmrgx_int)nvec, coef.data(), (dmrgx_int)ns, alpha.data(),
                                              beta.data(), norm2.data(), steps.data(), NULL);
            });
            if (ierr) return ierr;
            fprintf(f, ",\n    \"%s\": [", kind.name);
            for (PetscInt kx = 0; kx < Lx; ++kx) {
                fprintf(f, "%s\n      [", kx ? "," : "");
                for (PetscInt ky = 0; ky < Ly; ++ky) {
                    fprintf(f, "%s{", ky ? ",\n       " : "");
                    for (size_t part = 0; part < 2; ++part) {
                        const size_t v = 2 * (size_t)(kx * Ly + ky) + part;
                        fprintf(f, "%s\"%s\": {\"norm2\": %.17g, \"steps\": %lld, ", part ? ", " : "", part ? "sin" : "cos", norm2[v], LLD(steps[v]));
                        WriteAlphaBeta(f, &alpha[v * ns], &beta[v * ns], steps[v]);
                        fprintf(f, "}");
                    }
                    fprintf(f, "}");
                }
                fprintf(f, "]");
            }
            fprintf(f, "\n    ]");
        }
        spectral.EndRecord();
        return 0;
    }

    /** EXTENSION (-do_dynamical_correlations): one record of DynamicalCorrelations.json — the real-space dynamical correlation
        matrix from dmrgx_spectral_lanczos_overlaps.  Each source c (-dynamical_sources, default every site) starts one recurrence
        from O_c psi (coef row e_c) under the targets of CalculateSpectralFunction (zz: O = Sz under this step's H; pm: O = S- under
        the H of the sector qn - 1; mp: O = S+ under the H of qn + 1), and keeps the overlap of every Lanczos vector v_t with every
        site's panel O_s psi.  With T the tridiagonal matrix of alpha and beta and ‖O_c psi‖ = √norm2,
            <O_s psi| f(H) |O_c psi> = √norm2 Σ_t overlaps[t][s] f(T)_{t,0}
        exactly for f(H) = H^k, k < steps, and approximately for (z - H)^-1 (S_sc(ω) at z = ω + E0 + iη) and e^{-i(H - E0)τ}
        (G_sc(τ) = <S_s(τ) S_c>).  Written per operator as one entry per source: site, norm2, steps, the first `steps` of alpha
        and beta (beta[0] = 0) and `steps` rows of n overlaps.  At 12×6 with every site as a source and 64 steps a record holds
        about 3·72·64·72 numbers (some 20 MB); -dynamical_sources shrinks it in proportion. */
    PetscErrorCode CalculateDynamicalCorrelations(KronBlocks_t& KronBlocks, const ShellMat& H, const Vec& gsv_r, const PetscScalar E0, const Coords& r,
                                                  const std::vector<Hamiltonians::Term>& Terms, Block& SysBlockEnl, Block& EnvBlockEnl) {
        const PetscInt nsites = (PetscInt)r.x.size();
        const size_t n = r.x.size(), ns = (size_t)spectral_nsteps;
        std::vector<PetscInt> src = dyncorr_sources;
        if (src.empty())
            for (PetscInt s = 0; s < nsites; ++s) src.push_back(s);
        for (const PetscInt c : src)
            if (c >= nsites) SETERRQ2(mpi_comm, 1, "-dynamical_sources: site %lld is not in this %lld-site superblock.", LLD(c), LLD(nsites));
        const size_t nvec = src.size();
        std::vector<double> coef(nvec * n, 0.0);
        for (size_t v = 0; v < nvec; ++v) coef[v * n + (size_t)src[v]] = 1.0;
        FILE* f = dyncorr.BeginRecord(GlobIdx, LoopIdx);
        fprintf(f, ",\n    \"E0\": %.17g,\n    \"NSteps\": %lld", E0, LLD(spectral_nsteps));
        WriteSites(f, r);
        fprintf(f, ",\n    \"sources\": [");
        for (size_t v = 0; v < nvec; ++v) fprintf(f, "%s%lld", v ? ", " : "", LLD(src[v]));
        fprintf(f, "]");
        for (size_t k = 0; k < 3; ++k) {
            if (!spectral_ops[k]) continue;
            const SpectralKind& kind = spectral_kinds[k];
            std::vector<double> alpha(nvec * ns, 0.0), beta(nvec * ns, 0.0), norm2(nvec, 0.0), ov(nvec * ns * n, 0.0);
            std::vector<dmrgx_int> steps(nvec, 0);
            PetscErrorCode ierr = WithSpectralTarget(H, kind.op, Terms, SysBlockEnl, EnvBlockEnl, "dmrgx_spectral_lanczos_overlaps", [&](dmrgx_hshell t) {
                return dmrgx_spectral_lanczos_overlaps(KronBlocks.Handle(), gsv_r.d, t, kind.op, (dmrgx_int)nvec, coef.data(), (dmrgx_int)ns,
                                                       alpha.data(), beta.data(), norm2.data(), steps.data(), ov.data(), NULL);
            });
            if (ierr) return ierr;
            fprintf(f, ",\n    \"%s\": [", kind.name);
            for (size_t v = 0; v < nvec; ++v) {
                fprintf(f, "%s\n      {\"site\": %lld, \"norm2\": %.17g, \"steps\": %lld, ", v ? "," : "", LLD(src[v]), norm2[v], LLD(steps[v]));
                WriteAlphaBeta(f, &alpha[v * ns], &beta[v * ns], steps[v]);
                fprintf(f, ", \"overlaps\": [");
                for (dmrgx_int t = 0; t < steps[v]; ++t) {
                    fprintf(f, "%s\n        [", t ? "," : "");
                    const double* row = ov.data() + (v * ns + (size_t)t) * n;
                    for (size_t s = 0; s < n; ++s) fprintf(f, "%s%.17g", s ? ", " : "", row[s]);
                    fprintf(f, "]");
                }
                fprintf(f, "]}");
            }
            fprintf(f, "\n    ]");
        }
        dyncorr.EndRecord();
        return 0;
    }

    static std::string BlockDir(const std::string& BlockType, const PetscInt& iblock) { /* :2456-2464: "Sys_000000009/" */
        std::ostringstream oss; oss << BlockType << "_" << std::setfill('0') << std::setw(9) << iblock << "/"; return oss.str();
    }
    static std::string SweepDir(const PetscInt& isweep) { /* :2474-2481: "Sweep_000000002/" */
        std::ostringstream oss; oss << "Sweep_" << std::setfill('0') << std::setw(9) << isweep << "/"; return oss.str();
    }
    /** :2727-2764 — Hamiltonian.dat, PetscOptions.dat, Sweep.dat and (here) the blocks themselves, at the end of a completed loop */
    PetscErrorCode SaveSweepsData() {
        if (!do_save_blocks) return 0;
        /* The blocks are replicated on every rank of a multi-GPU run: rank 0 alone writes the checkpoint (every rank writing
           the same files would truncate what another had finished, and cost N device-to-host gathers). */
        { int rank = 0, world = 1; dmrgx_ctx_rank(DmrgxContext(), &rank, &world); if (rank != 0) return 0; }
        PetscErrorCode ierr;
        int spin_type_key = 102; /* SpinOneHalf = 102, SpinOne = 101 (include/DMRGBlock.hpp:51-55) */
        { std::string sp; PetscBool set; PetscOptions::DB().GetString("-spin", sp, &set); if (set && sp == "1") spin_type_key = 101; }
        const std::string dir = scratch_dir + SweepDir(LoopIdx);
        ierr = Makedir(dir); CHKERRQ(ierr);
        /* Sweep.dat is the commit marker -restart_dir looks for: an older one in this directory goes first, the new one is
           written to a temporary name, flushed to disk and renamed into place after every block file is complete. */
        remove((dir + "Sweep.dat").c_str());
        for (PetscInt iblock = 0; iblock < sys_ninit; ++iblock) {
            if (!sys_blocks[(size_t)iblock].Initialized()) continue;
            ierr = BlockIO::Save(sys_blocks[(size_t)iblock], dir + BlockDir("Sys", iblock), io_int_bytes, spin_type_key); CHKERRQ(ierr);
        }
        ierr = Ham.SaveAsOptions(dir + "Hamiltonian.dat"); CHKERRQ(ierr);
        {
            std::ofstream f((dir + "PetscOptions.dat").c_str());
            for (const char* key : {"-spin", "-mstates", "-mwarmup", "-nsweeps", "-msweeps", "-maxnsweeps"}) {
                std::string v; PetscBool set;
                PetscOptions::DB().GetString(key, v, &set);
                if (set) f << key << " " << (v.empty() ? "yes" : v) << std::endl;
            }
        }
        const std::string tmp = dir + "Sweep.dat.tmp";
        {
            FILE* f = fopen(tmp.c_str(), "w");
            if (!f) SETERRQ1(mpi_comm, 1, "cannot write %s", tmp.c_str());
            const PetscInt num_env_blocks = 1, env_ninit = 0;
#define SWEEP_DUMP(VAR) fprintf(f, "%20s  %lld\n", #VAR, (long long)(VAR));
            SWEEP_DUMP(GlobIdx); SWEEP_DUMP(LoopIdx); SWEEP_DUMP(num_sys_blocks); SWEEP_DUMP(num_env_blocks); SWEEP_DUMP(sys_ninit); SWEEP_DUMP(env_ninit);
            SWEEP_DUMP(num_sites); SWEEP_DUMP(sweep_mode); SWEEP_DUMP(msweep_idx);
#undef SWEEP_DUMP
            fflush(f);
            fsync(fileno(f));
            fclose(f);
        }
        sync(); /* the block files reach the disk before the marker names them */
        if (rename(tmp.c_str(), (dir + "Sweep.dat").c_str())) SETERRQ1(mpi_comm, 1, "cannot commit %sSweep.dat", dir.c_str());
        return 0;
    }

    /** :2484-2513 */
    PetscErrorCode SaveStepHeaders() {
        fprintf(fp_step, "{\n  \"headers\" : [");
        const char* h[] = {"GlobIdx", "LoopType", "LoopIdx", "StepIdx", "NSites_Sys", "NSites_Env", "NSites_SysEnl", "NSites_EnvEnl", "NStates_Sys",
                           "NStates_Env", "NStates_SysEnl", "NStates_EnvEnl", "NStates_SysRot", "NStates_EnvRot", "NumStates_H", "TruncErr_Sys",
                           "TruncErr_Env", "GSEnergy"};
        for (int i = 0; i < 18; ++i) fprintf(fp_step, "\"%s\"%s", h[i], i < 17 ? ", " : "");
        fprintf(fp_step, "  ],\n  \"table\" : ");
        fflush(fp_step);
        return 0;
    }
    /** :2516-2566 (tabular form, the reference's default) */
    PetscErrorCode SaveStepData(const StepData& d) {
        fprintf(fp_step, "%s", rows_written ? ",\n" : ""); /* (the reference keys the comma on GlobIdx, which breaks the file after a restart) */
        fprintf(fp_step, "    [ %lld, %s, %lld, %lld, ", LLD(GlobIdx), LoopType ? "\"Sweep\"" : "\"Warmup\"", LLD(LoopIdx), LLD(StepIdx));
        fprintf(fp_step, "%lld, %lld, %lld, %lld, ", LLD(d.NumSites_Sys), LLD(d.NumSites_Env), LLD(d.NumSites_SysEnl), LLD(d.NumSites_EnvEnl));
        fprintf(fp_step, "%lld, %lld, %lld, %lld, ", LLD(d.NumStates_Sys), LLD(d.NumStates_Env), LLD(d.NumStates_SysEnl), LLD(d.NumStates_EnvEnl));
        fprintf(fp_step, "%lld, %lld, %lld, ", LLD(d.NumStates_SysRot), LLD(d.NumStates_EnvRot), LLD(d.NumStates_H));
        fprintf(fp_step, "%.12g, %.12g, %.12g]", d.TruncErr_Sys, d.TruncErr_Env, d.GSEnergy);
        fflush(fp_step);
        return 0;
    }
    /** :2568-2616 */
    PetscErrorCode SaveTimingsHeaders() {
        fprintf(fp_timings, "{\n  \"headers\" : [\"GlobIdx\", \"Total\", \"Enlr\", \"Kron\", \"Diag\", \"Rdms\", \"Rotb\" ],\n  \"table\" : ");
        fflush(fp_timings);
        return 0;
    }
    PetscErrorCode SaveTimingsData(const TimingsData& d) {
        fprintf(fp_timings, "%s", rows_written ? ",\n" : "");
        fprintf(fp_timings, "    [ %lld, %.9g, %.9g, %.9g, %.9g, %.9g, %.9g ]", LLD(GlobIdx), d.Total, d.tEnlr, d.tKron, d.tDiag, d.tRdms, d.tRotb);
        fflush(fp_timings);
        return 0;
    }
    /** :2618-2665 — the unsorted, per-block-grouped spectra (what GetTruncation hands over at :1790-1793) */
    PetscErrorCode SaveEntanglementSpectra(const BasisTransformation& L, const std::vector<PetscReal>& qn_L, const BasisTransformation& R,
                                           const std::vector<PetscReal>& qn_R) {
        fprintf(fp_entanglement, "%s", rows_written ? ",\n" : "");
        fprintf(fp_entanglement, "  {\n    \"GlobIdx\": %lld,\n", LLD(GlobIdx));
        const BasisTransformation* bt[2] = {&L, &R};
        const std::vector<PetscReal>* qn[2] = {&qn_L, &qn_R};
        const char* label[2] = {"Sys", "Env"};
        for (int s = 0; s < 2; ++s) {
            dmrgx_int mm, n, ns, ne; double te;
            DMRGX_CALL(dmrgx_xform_info(bt[s]->h, &mm, &n, &ns, &te, &ne));
            std::vector<double> ev((size_t)ne); std::vector<dmrgx_int> bi((size_t)ne);
            DMRGX_CALL(dmrgx_xform_spectrum(bt[s]->h, ev.data(), bi.data()));
            fprintf(fp_entanglement, "    \"%s\": [\n", label[s]);
            dmrgx_int prev = 999999999;
            for (dmrgx_int k = 0; k < ne; ++k) {
                if (prev != bi[(size_t)k]) {
                    if (prev != 999999999) fprintf(fp_entanglement, " ]},\n");
                    fprintf(fp_entanglement, "      {\"sector\": %g, \"vals\": [ %g", (*qn[s])[(size_t)bi[(size_t)k]], ev[(size_t)k]);
                } else fprintf(fp_entanglement, ", %g", ev[(size_t)k]);
                prev = bi[(size_t)k];
            }
            fprintf(fp_entanglement, " ]}\n    ]%s\n", s == 0 ? "," : "");
        }
        fprintf(fp_entanglement, "  }");
        fflush(fp_entanglement);
        return 0;
    }
    /** :2668-2686 (+ seconds per sweep and the H*psi count, which the reference leaves to Timings.json) */
    PetscErrorCode SaveLoopsData() {
        fprintf(fp_data, ",\n  \"Warmup\": {\n    \"MStates\": %lld\n  },\n  \"Sweeps\": {\n    \"MStates\": [", LLD(mwarmup));
        for (size_t i = 0; i < sweeps_mstates.size(); ++i) fprintf(fp_data, "%s %lld", i ? "," : "", LLD(sweeps_mstates[i]));
        fprintf(fp_data, " ],\n    \"Seconds\": [");
        for (size_t i = 0; i < sweeps_seconds.size(); ++i) fprintf(fp_data, "%s %.9g", i ? "," : "", sweeps_seconds[i]);
        fprintf(fp_data, " ]\n  },\n  \"NumMatVecs\": %lld,\n  \"MatVecFlops\": %.6g,\n  \"StepsWithPredictedStart\": %lld", LLD(total_matvecs), total_matvec_flops, steps_predicted);
        fflush(fp_data);
        return 0;
    }

    MPI_Comm mpi_comm = PETSC_COMM_SELF;
    PetscBool init = PETSC_FALSE, verbose = PETSC_FALSE, dry_run = PETSC_FALSE, warmed_up = PETSC_FALSE, no_symm = PETSC_FALSE, do_shell = PETSC_TRUE;
    PetscReal qn_sector = 0.0;
    SweepMode_t sweep_mode = SWEEP_MODE_NULL;
    PetscInt mwarmup = 0, nsweeps = 0;
    std::vector<PetscInt> msweeps, maxnsweeps, sweeps_mstates;
    std::vector<double> sweeps_seconds;
    PetscInt msweep_idx = -1;
    PetscInt num_sites = 0, num_sys_blocks = 0;
    std::vector<Block> sys_blocks;
    PetscInt sys_ninit = 0;
    Hamiltonian Ham;
    Block SingleSite;
    Block& AddSite = SingleSite;
    std::string scratch_dir = ".", restart_dir;
    PetscBool restart = PETSC_FALSE, do_save_blocks = PETSC_FALSE;
    int io_int_bytes = 4;
    static const PetscInt MAX_SWEEP_IDX = 10000;
    FILE *fp_step = NULL, *fp_timings = NULL, *fp_entanglement = NULL, *fp_data = NULL, *fp_corr = NULL;
    PetscInt GlobIdx = 0;
    Step_t LoopType = NullStep;
    PetscInt LoopIdx = 0, StepIdx = 0;
    std::vector<Correlator> measurements;
    PetscBool corr_headers_printed = PETSC_FALSE, corr_printed_first = PETSC_FALSE;
    /* the extensions' output files; one that is not open means the extension is off */
    RecordFile corrmat;                       /* -do_correlation_matrix */
    RecordFile dimer;                         /* -do_dimer_matrix */
    RecordFile spectral;                      /* -do_spectral_function */
    RecordFile dyncorr;                       /* -do_dynamical_correlations */
    PetscInt spectral_nsteps = 64;            /* -spectral_nsteps */
    std::vector<bool> spectral_ops = {true, true, true}; /* -spectral_ops, in the order of spectral_kinds */
    std::vector<PetscInt> dyncorr_sources;    /* -dynamical_sources; empty: every site */
    PetscScalar gse = 0.0;
    std::vector<PetscReal> trunc_err;
    double t0abs = 0.0;
    dmrgx_eigs_opts eps_opts = {1e-8, 16, 0, 20261018ULL}; /* SLEPc defaults: tol 1e-8, ncv 16 */
    /* -wavefunction_prediction (extension): per block the transformation that created it and the serial of the block it enlarged */
    PetscBool do_prediction = PETSC_FALSE;
    std::vector<std::shared_ptr<BasisTransformation>> sys_bt;
    std::vector<long long> sys_bt_src;
    struct PendingWaves {
        dmrgx_wave wL = nullptr, wR = nullptr;
        long long out_sys = -1, out_env = -1, xe_left_src = -2, xe_right_src = -2;
        std::shared_ptr<BasisTransformation> xe_left, xe_right;
    } pending;
    long long steps_predicted = 0;
    void ClearPendingWaves() {
        if (pending.wL) dmrgx_wave_destroy(pending.wL);
        if (pending.wR) dmrgx_wave_destroy(pending.wR);
        pending = PendingWaves();
    }
    long long BlockIndex(const Block& b) const {
        if (sys_blocks.empty() || &b < sys_blocks.data() || &b >= sys_blocks.data() + sys_blocks.size()) return -1;
        return (long long)(&b - sys_blocks.data());
    }
    long long total_matvecs = 0, rows_written = 0;
    double total_matvec_flops = 0;
};
