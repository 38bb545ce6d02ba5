/*  DMRG-SquareLattice — the reference's executable (src/DMRG-SquareLattice.cpp:16-181) over the B200 path.
 *
 *      DMRG-SquareLattice.x -Lx 12 -Ly 6 -J1 0.5 -Jz1 1 -J2 0.25 -Jz2 0.5 -mwarmup 128 -msweeps 512,1024,2048 \
 *                           [-H_eps_tol 1e-12] [-data_dir out/] [-device 0] [-verbose] [-wavefunction_prediction 1] [-do_correlation_matrix 1]
 *                           [-do_dimer_matrix 1]
 *
 *  Same options (plus -device and the opt-in -wavefunction_prediction, -do_correlation_matrix and -do_dimer_matrix, which the reference does not have), same stdout banner, same JSON files; one process drives one B200 through the C ABI
 *  (include/dmrgx.h).  There is no CPU path: without a CUDA device the context creation fails and the
 *  program exits non-zero.
 */
static char help[] = "DMRG executable for the Spin-1/2 J1-J2 XY Model on a two-dimensional square lattice (B200 path).\n"
                     "Extensions, off by default, computed and written by rank 0 at every measurement step:\n"
                     "  -do_correlation_matrix 1   every <S_i S_j> and the structure factor S(q) -> CorrelationMatrix.json\n"
                     "  -do_dimer_matrix 1         <D_a>, <D_a D_b> over the nearest-neighbour bonds (D_a = S_i.S_j) and the\n"
                     "                             dimer structure factors of the x and y bonds -> DimerMatrix.json\n";

#include <unistd.h>

#include "DMRGBlock.hpp"
#include "DMRGBlockContainer.hpp"
#include "Hamiltonians.hpp"

typedef DMRGBlockContainer<Block::SpinBase, Hamiltonians::J1J2XXZModel_SquareLattice> DMRG_t;
PetscErrorCode Correlators(DMRG_t& DMRG);

int main(int argc, char** argv) {
    PetscErrorCode ierr;
    PetscOptions& o = PetscOptions::DB();
    o.Insert(argc, argv);
    if (o.Has("-help") || o.Has("-h")) { printf("%s", help); return 0; }
    { /* -options_file like PetscOptionsInsertFile */
        std::string f; PetscBool set;
        o.GetString("-options_file", f, &set);
        if (set) {
            std::ifstream in(f);
            if (!in) { fprintf(stderr, "cannot read -options_file %s\n", f.c_str()); return 1; }
            std::stringstream ss; ss << in.rdbuf();
            o.InsertString(ss.str());
            o.Insert(argc, argv); /* the command line wins */
        }
    }
    /* One process per GPU.  Launched by `python -m torch.distributed.run --no-python --nproc-per-node N …` (or any launcher
       that sets RANK / WORLD_SIZE / LOCAL_RANK): rank 0 creates the communicator id and passes it on through a file, every
       rank drives the GPU of its LOCAL_RANK, and only rank 0 prints and writes the JSON files of -data_dir. */
    auto env_int = [](const char* k, int dflt) { const char* v = getenv(k); return v ? atoi(v) : dflt; };
    const int rank = env_int("RANK", 0), world = env_int("WORLD_SIZE", 1);
    PetscInt device = env_int("LOCAL_RANK", 0);
    o.GetInt("-device", &device, NULL);
    if (world > 1) {
        unsigned char id[128];
        const char* idf = getenv("DMRGX_ID_FILE");
        const std::string id_file = idf ? idf : std::string("/tmp/dmrgx_id_") + (getenv("MASTER_PORT") ? getenv("MASTER_PORT") : "0");
        if (rank == 0) {
            if (dmrgx_dist_unique_id(id)) { fprintf(stderr, "[dmrgx] %s\n", dmrgx_last_error()); return 110; }
            FILE* f = fopen((id_file + ".tmp").c_str(), "wb");
            if (!f || fwrite(id, 1, 128, f) != 128) { fprintf(stderr, "cannot write %s\n", id_file.c_str()); return 1; }
            fclose(f);
            rename((id_file + ".tmp").c_str(), id_file.c_str());
        } else {
            FILE* f = nullptr;
            for (int tries = 0; tries < 6000 && !(f = fopen(id_file.c_str(), "rb")); ++tries) usleep(10000);
            if (!f || fread(id, 1, 128, f) != 128) { fprintf(stderr, "rank %d: cannot read the communicator id from %s\n", rank, id_file.c_str()); return 1; }
            fclose(f);
            if (!freopen("/dev/null", "w", stdout)) return 1;
            std::string dd = "./data_dir/"; PetscBool set;
            o.GetString("-data_dir", dd, &set);
            o.kv["-data_dir"] = dd + (dd.back() == '/' ? "" : "/") + ".rank" + std::to_string(rank) + "/";
        }
        if (dmrgx_ctx_create_dist((int)device, NULL, rank, world, id, &DmrgxContext())) { fprintf(stderr, "[dmrgx] %s\n", dmrgx_last_error()); return 100; }
        if (rank == 0) remove(id_file.c_str()); /* the communicator exists: every rank has read it */
    } else if (dmrgx_ctx_create((int)device, NULL, &DmrgxContext())) {
        fprintf(stderr, "[dmrgx] %s\n", dmrgx_last_error());
        return 100;
    }
    {
        DMRG_t DMRG(PETSC_COMM_WORLD);
        ierr = DMRG.Initialize(); CHKERRQ(ierr);
        PetscBool do_corr = PETSC_TRUE;
        o.GetBool("-do_correlators", &do_corr, NULL);
        if (do_corr) { ierr = Correlators(DMRG); CHKERRQ(ierr); }
        ierr = DMRG.Warmup(); CHKERRQ(ierr);
        ierr = DMRG.Sweeps(); CHKERRQ(ierr);
        printf("Final ground state energy: %.12f   kernel launches: %lld\n", DMRG.GroundStateEnergy(), dmrgx_launch_count());
        ierr = DMRG.Destroy(); CHKERRQ(ierr);
    }
    dmrgx_ctx_destroy(DmrgxContext());
    return 0;
}

static std::string SiteLabel(const DMRG_t& DMRG, Op_t t, PetscInt idx) {
    PetscInt ix, jy;
    DMRG.HamiltonianRef().To2D(idx, ix, jy);
    return OpToStr(t) + "_{" + std::to_string(ix) + "," + std::to_string(jy) + "} ";
}

/** The measurements of src/DMRG-SquareLattice.cpp:40-181: site magnetisations, nearest-neighbour bond correlators
    (Sz-Sz, Sp-Sm, Sm-Sp), one row, two columns (Polyakov loops) and the interior Wilson loop. */
PetscErrorCode Correlators(DMRG_t& DMRG) {
    PetscErrorCode ierr;
    const PetscInt Lx = DMRG.HamiltonianRef().Lx(), Ly = DMRG.HamiltonianRef().Ly();
    const PetscInt NumSitesSys = Lx * Ly / 2;
    for (PetscInt idx = 0; idx < NumSitesSys; ++idx) {
        ierr = DMRG.SetUpCorrelation({{OpSz, idx}}, "Magnetization(" + std::to_string(idx) + ")", "< " + SiteLabel(DMRG, OpSz, idx) + ">"); CHKERRQ(ierr);
    }
    for (const std::vector<PetscInt>& pair : DMRG.HamiltonianRef().NeighborPairs()) {
        if (pair.size() != 2) SETERRQ1(PETSC_COMM_WORLD, 1, "Invalid 2-point correlator. Got %lld operators instead.", LLD(pair.size()));
        const Op_t types[3][2] = {{OpSz, OpSz}, {OpSp, OpSm}, {OpSm, OpSp}};
        for (const auto& ty : types) {
            std::vector<Op> OpList;
            std::string desc = "< ", name = std::string("NearestNeighbor") + OpToStr(ty[0]) + OpToStr(ty[1]) + "( ";
            for (int i = 0; i < 2; ++i) {
                OpList.push_back({ty[i], pair[(size_t)i]});
                desc += SiteLabel(DMRG, ty[i], pair[(size_t)i]);
                name += std::to_string(pair[(size_t)i]) + " ";
            }
            ierr = DMRG.SetUpCorrelation(OpList, name + ")", desc + ">"); CHKERRQ(ierr);
        }
    }
    auto loop = [&](const std::vector<std::pair<PetscInt, PetscInt>>& xy, const std::string& name) -> PetscErrorCode {
        std::vector<Op> OpList;
        std::string desc = "< ";
        for (auto& p : xy) {
            const PetscInt idx = DMRG.HamiltonianRef().To1D(p.first, p.second);
            OpList.push_back({OpSz, idx});
            desc += "Sz_{" + std::to_string(p.first) + "," + std::to_string(p.second) + "} ";
        }
        return DMRG.SetUpCorrelation(OpList, name, desc + ">");
    };
    std::vector<std::pair<PetscInt, PetscInt>> xy;
    for (PetscInt i = 0; i < Lx; ++i) xy.push_back({i, 1});
    ierr = loop(xy, "MagnetizationRowX1"); CHKERRQ(ierr);
    xy.clear(); for (PetscInt j = 0; j < Ly; ++j) xy.push_back({1, j});
    ierr = loop(xy, "Polyakov"); CHKERRQ(ierr);
    xy.clear(); for (PetscInt j = 0; j < Ly; ++j) xy.push_back({Lx - 2, j});
    ierr = loop(xy, "Polyakov2"); CHKERRQ(ierr);
    xy.clear();
    for (PetscInt j = 1; j < Ly - 2; ++j) xy.push_back({1, j});
    for (PetscInt i = 1; i < Lx - 2; ++i) xy.push_back({i, Ly - 2});
    for (PetscInt j = Ly - 2; j > 1; --j) xy.push_back({Lx - 2, j});
    for (PetscInt i = Lx - 2; i > 1; --i) xy.push_back({i, 1});
    ierr = loop(xy, "Wilson"); CHKERRQ(ierr);
    return 0;
}
