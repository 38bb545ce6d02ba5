/*  common.h — host-side object model of the B200 superblock path.
 *
 *  Mirrors the reference's types at the granularity the hot path needs:
 *    Sectors  <-> QuantumNumbers            (include/QuantumNumbers.hpp:30-239)
 *    Block    <-> Block::SpinBase           (include/DMRGBlock.hpp:79-434)
 *    Kron     <-> KronBlocks_t              (include/DMRGKron.hpp:117-480)
 *    HShell   <-> KronSumShellCtx + MatMult_KronSumShell (include/DMRGKron.hpp:92-112, src/DMRGKron.cpp:1827-1869)
 *    XForm    <-> BasisTransformation       (include/DMRGBlockContainer.hpp:226-257)
 *  but laid out for HBM: an operator is not a CSR matrix, it is a list of TILES per sector block —
 *  dense FP64 panels (after truncation), CSR panels (exact blocks) or scaled identities (added-site
 *  operators 1⊗s) — so that A·X·Bᵀ per sector pair becomes a short chain of dense panel products.
 */
#pragma once
#include <cstdint>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "dev.h"

namespace dmrgx {

/* PETSc error codes the reference returns on this path (petscerror.h, 3.8) */
enum { OK = 0, ERR_GENERIC = 1, ERR_SUP = 56, ERR_ARG_WRONG = 62, ERR_ARG_OUTOFRANGE = 63, ERR_ARG_CORRUPT = 64, ERR_ARG_WRONGSTATE = 73,
       ERR_NO_DEVICE = 100 };

struct Err : std::runtime_error {
    int code;
    Err(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

/* include/DMRGBlock.hpp:21-27 */
enum { OP_SM = -1, OP_SZ = 0, OP_SP = 1, OP_EYE = 2, OP_H = 3 };

struct Ctx {
    dev::Stream* st = nullptr;
    int rank = 0, world = 1;
    double dense_fill_threshold = 0.125; /* sector-block tiles with fill >= this are stored dense */
};

/* ref-counted device allocation */
struct DevBuf {
    Ctx* ctx;
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf(Ctx* c, size_t b) : ctx(c), bytes(b) { p = dev::malloc_bytes(c->st, b); }
    ~DevBuf() { dev::free_bytes(ctx->st, p); }
    DevBuf(const DevBuf&) = delete;
    template <class T> T* as() const { return (T*)p; }
};
typedef std::shared_ptr<DevBuf> BufRef;

struct Sectors {
    std::vector<double> qn;
    std::vector<int> size, off; /* off has nsec+1 entries */
    int nsec() const { return (int)qn.size(); }
    int nstates() const { return off.empty() ? 0 : off.back(); }
    void init(const std::vector<double>& q, const std::vector<long long>& s);
    int sector_of(int idx) const;
};

enum TileFmt : int { T_DENSE = 0, T_CSR = 1, T_EYE = 2 };

/* host copy of the packed CSR arrays of one uploaded operator (small: exact, un-truncated blocks only) — the sparse
   shell planner flattens them per sector without reading them back from the device */
struct HostCsr { std::vector<int> rowptr, col; std::vector<double> val; };

/* A rectangular piece of one sector block (I, I+shift) of an operator, in GLOBAL block coordinates. */
struct Tile {
    int r0 = 0, c0 = 0, nr = 0, nc = 0;
    TileFmt fmt = T_DENSE;
    /* DENSE: element (i,j) = d[i*sr + j*sc]  (sr,sc) = (ld,1) row-major or (1,ld) for a transposed view */
    const double* d = nullptr;
    long long sr = 0, sc = 0;
    /* CSR: local indices, nr rows */
    const int* rowptr = nullptr;
    const int* col = nullptr;
    const double* val = nullptr;
    long long nnz = 0;
    std::shared_ptr<const HostCsr> hcsr; /* CSR: row i of this tile = entries [hcsr->rowptr[h_rp+i], hcsr->rowptr[h_rp+i+1]) of */
    long long h_rp = 0, h_ci = 0;        /*      hcsr->col / val starting at h_ci (the same numbers the device arrays hold)   */
    /* DENSE tiles of at most 256x256 that came from the host keep a host copy too (the small, filled sector blocks at the edge
       of an otherwise sparse exact block): element (i,j) = (*hdense)[h_d0 + i*sr + j*sc] */
    std::shared_ptr<const std::vector<double>> hdense;
    long long h_d0 = 0;
    /* EYE: scale * I_nr */
    double scale = 1.0;
    BufRef owner;
    long long bytes() const { /* algorithmic bytes of this tile (SURVEY §8d) */
        if (fmt == T_DENSE) return 8LL * nr * nc;
        if (fmt == T_CSR) return 12LL * nnz + 4LL * (nr + 1);
        return 0;
    }
};

struct Operator {
    int shift = 0;                         /* column sector = row sector + shift */
    std::vector<std::vector<Tile>> tiles;  /* per row sector */
    bool present = false;
};

struct Block {
    Ctx* ctx = nullptr;
    int nsites = 0;
    Sectors sec;
    std::vector<Operator> Sz, Sp, Sm; /* Sm[i] = Sp[i]^T as transposed views (src/DMRGBlock.cpp:623-636) */
    Operator H;
    const Operator* op(int optype, int isite) const;
};

struct Term { double a; int Iop; long long Isite; int Jop; long long Jsite; }; /* include/Hamiltonians.hpp:17-24 */

struct KronPair { double qn; int il, ir, size; };

struct Kron {
    Ctx* ctx = nullptr;
    const Block* L = nullptr;
    const Block* R = nullptr;
    std::vector<KronPair> pairs;
    std::vector<long long> off; /* npairs+1 */
    std::map<std::pair<int, int>, int> map;
    long long nstates() const { return off.back(); }
    int find(int il, int ir) const { auto f = map.find({il, ir}); return f == map.end() ? -1 : f->second; }
};

struct Plan {
    std::vector<dev::WorkItem> items;
    std::vector<dev::Segment> segs;
    std::vector<dev::ReduceItem> reduces;   /* split chains: partial tiles in the scratch, summed in a second launch */
    long long scratch_elems = 0;
    /* when > 0, emit_cells cuts chains whose cost (sum of K) times tile area exceeds this many multiply-adds */
    double split_item_cost = 0;
    /* launch order: items are sorted by (phase, cost descending).  Stage 2 of the shell sets phase = index of the chain part,
       so that the CTAs resident at any time work on the same range of left-operator groups: their V and right-factor
       panels (a fraction of the 270 + 93 MB at 12x6 m = 2048) then fit in L2 together instead of being re-read. */
    std::vector<int> item_phase;
    BufRef d_items, d_segs, d_reduces, scratch;
    void upload(Ctx* ctx);
    void run(Ctx* ctx, const double* x = nullptr, double* y = nullptr) const;
    /* useful work of the plan: 2*M*N*K of GEMM segments actually inside tile extents */
    double flops = 0;
    double exec_flops = 0; /* what the kernel executes for them: padded to whole fragments and K chunks */
};

/* The sparse-sector form of the shell (north_star (a): un-truncated blocks whose operators are CSR / scaled-identity
   tiles): ONE fused launch of spmm_kernel per apply instead of the two chain launches. */
struct SparsePlan {
    std::vector<dev::SpTile> tiles;
    std::vector<dev::SpASlot> aslots;    /* the row programs, slot-major per tile */
    std::vector<dev::SpSSlot> sslots;
    std::vector<dev::SpBSlot> bslots;
    BufRef d_tiles, d_aslots, d_sslots, d_bslots, d_int, d_val;
    int max_nR = 0;
    double flops = 0;
};

struct HShell {
    Ctx* ctx = nullptr;
    const Kron* kron = nullptr;
    long long n = 0;
    /* superblock rows this rank computes ([0,n) on one GPU) and the ownership table of all ranks (world+1 entries) */
    long long row_begin = 0, row_end = 0;
    std::vector<long long> row_cuts;
    /* sector halo of the sharded apply (SURVEY.md §8e): the point-to-point transfers that bring every rank the X_q panels its
       tiles read and nothing else — the same list on every rank */
    std::vector<int> halo_from, halo_to;
    std::vector<long long> halo_off, halo_cnt;
    long long halo_recv_elems = 0;   /* what this rank receives per apply */
    Plan stage1, stage2;
    std::unique_ptr<SparsePlan> sparse; /* when set, the apply is one spmm launch and stage1 / stage2 are empty */
    BufRef work;                 /* V panels of stage 1 */
    BufRef xbuf, ybuf;           /* device staging of the host-buffer entry point */
    std::vector<BufRef> keep;    /* pre-summed right factors etc. */
    std::vector<std::shared_ptr<Operator>> keep_ops; /* operator products of correlators */
    long long alg_bytes = 0;     /* SURVEY §8d: 16*D + distinct operator tile bytes */
    double alg_flops = 0;
    long long alg_bytes_global = 0; /* the same two figures for the whole (unsharded) operator */
    double alg_flops_global = 0;
    int nterms = 0;
};

struct XForm {
    Ctx* ctx = nullptr;
    Sectors newsec;                      /* kept sectors */
    std::vector<int> old_sector;         /* new sector index -> old (enlarged) sector index */
    std::vector<int> old_off, old_size;  /* offset / size of that old sector in the enlarged basis */
    std::vector<BufRef> U;               /* per new sector: m_I × n_I row-major, rows = kept eigenvectors (descending) */
    double trunc_err = 0;
    std::vector<double> spec_eig;        /* grouped (unsorted) spectrum as dumped to EntanglementSpectra.json */
    std::vector<int> spec_blk;
    int nstates_old = 0;
};

/* This step's ground state with the growing side already projected onto its kept states (predict.cpp) */
struct Wave {
    Ctx* ctx = nullptr;
    bool grow_left = true;
    Sectors grown;                   /* sectors of the new block on the growing side */
    std::vector<double> other_qn;    /* sectors of the old ENLARGED block on the other side */
    std::vector<int> other_size;
    struct Blk { int kg, io; long long off, src; }; /* kept sector of the grown side, enlarged sector of the other side */
    std::vector<Blk> blks;
    BufRef phi;
};

/* DMRGX_TRACE=1: wall-clock of the sub-phases of the host-side orchestration (device drained at each mark), to stderr */
struct Trace {
    Ctx* ctx; const char* what; double t0; bool on;
    static bool enabled();
    static double now();
    Trace(Ctx* c, const char* w);
    void mark(const char* label);
};

/* ---- functions implemented across the .cpp files ---- */
Block* block_from_csr_begin(Ctx*, int nsites, const std::vector<double>& qn, const std::vector<long long>& sizes);
void block_set_operator(Block*, int optype, int isite, const long long* rowptr, const long long* col, const double* val);
void block_get_operator(const Block*, int optype, int isite, std::vector<long long>& rowptr, std::vector<long long>& col,
                        std::vector<double>& val);
Block* block_single_site(Ctx*, int spin_twice);
Block* block_enlarge(const Block* L, const Block* site, const std::vector<Term>& terms);
void block_check(const Block*);

std::vector<Term> ham_terms(long long Lx, long long Ly, double J1, double Jz1, double J2, double Jz2, int bcx, int bcy, long long nsites);

Kron* kron_create(const Block* L, const Block* R, const std::vector<double>& qn_sectors);

HShell* hshell_create(const Kron*, const std::vector<Term>& terms);
HShell* hshell_create_single(const Kron*, int opl, int il, int opr, int ir);
HShell* hshell_create_product(const Kron*, const std::vector<std::pair<int, int>>& lops, const std::vector<std::pair<int, int>>& rops);
void hshell_apply(HShell*, const double* d_x, double* d_y);
void hshell_apply_sharded(HShell*, double* d_x, double* d_y);

struct EigsOpts { double tol = 1e-8; int ncv = 16; int max_it = 0; unsigned long long seed = 20261018ULL; };
struct EigsStats { long long nmatvec = 0, nrestart = 0; double resid = 0; int converged = 0; };
/* d_init: optional start vector of the global length (device; every rank holds all of it), else a seeded random one */
double eigs_smallest(HShell*, const EigsOpts&, double* d_psi, EigsStats*, const double* d_init = nullptr);

void truncate(const Kron*, const double* d_psi, long long mstates, XForm** L, XForm** R);
Block* rotate(const Block* enl, const XForm* xf);

/* predict.cpp: wave-function transformation (extension; the reference always starts from a random vector) */
Wave* wave_create(const Kron*, const double* d_psi, const XForm* grown_side, bool grow_left);
bool wave_apply(const Wave*, const XForm* shrinking_side, const Block* site, const Kron* new_kron, double* d_psi_new);

/* corr.cpp: all two-point spin correlators of the superblock (extension; host n×n outputs, n = sites of both blocks) */
void corr_matrix(const Kron*, const double* d_psi, double* szsz, double* spsm, double* smsp, double* sz, double* flops);
/* corr.cpp: the bond–bond correlators of nb isotropic bonds (extension; host nb×nb and nb outputs) */
void dimer_matrix(const Kron*, const double* d_psi, long long nb, const long long* bond_i, const long long* bond_j, double* dd, double* d,
                  double* flops);
/* corr.cpp: continued-fraction (Lanczos) coefficients of nvec start vectors Σ_s coef_s O_s psi under the target shell (extension);
   overlaps (nvec × nsteps × n, may be NULL): <O_s psi, v_t> of every Lanczos vector with every single-site panel */
void spectral_lanczos(const Kron*, const double* d_psi, HShell* h_target, int op, long long nvec, const double* coef, long long nsteps,
                      double* alpha, double* beta, double* norm2, long long* nsteps_done, double* overlaps, double* flops);

}  // namespace dmrgx
