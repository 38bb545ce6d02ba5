/*  dmrgx.h — C ABI of the B200-native superblock-diagonalisation path of DMRG.x.
 *
 *  This is the drop-in boundary: each entry point replaces one piece of the reference's hot path and
 *  cites it (paths relative to the reference tree).  A maintainer of the reference binds these from
 *  KronBlocks_t / Block::SpinBase / DMRGBlockContainer (see INTEGRATION.md for the stubs).
 *
 *  Conventions (SURVEY.md §8b)
 *    - every function returns an int status, 0 = success; non-zero values reuse the PETSc error codes
 *      the reference returns on this path (63 PETSC_ERR_ARG_OUTOFRANGE, 62 PETSC_ERR_ARG_WRONG,
 *      73 PETSC_ERR_ARG_WRONGSTATE, 64 PETSC_ERR_ARG_CORRUPT, 56 PETSC_ERR_SUP, 1 generic,
 *      100+ = CUDA / no device).  dmrgx_last_error() gives the message.  No exception crosses the ABI.
 *    - opaque handles; the library owns all device memory; the caller owns host buffers; every
 *      *_create / *_upload has a matching *_destroy.  One driving host thread per context.
 *    - index type is 64-bit (`dmrgx_int`), matching a 64-bit-PetscInt build; operator enum values are
 *      the reference's Op_t (include/DMRGBlock.hpp:21-27) and double as the Sz sector shift.
 *    - there is NO CPU path: dmrgx_ctx_create fails with 100 when no CUDA device is present.
 */
#ifndef DMRGX_H
#define DMRGX_H

#ifdef __cplusplus
extern "C" {
#endif

typedef long long dmrgx_int;

typedef struct dmrgx_ctx_s* dmrgx_ctx;
typedef struct dmrgx_block_s* dmrgx_block;
typedef struct dmrgx_kron_s* dmrgx_kron;
typedef struct dmrgx_hshell_s* dmrgx_hshell;
typedef struct dmrgx_xform_s* dmrgx_xform;

/* include/DMRGBlock.hpp:21-27 (+ H, which the reference keeps as a separate Mat member) */
enum { DMRGX_OP_SM = -1, DMRGX_OP_SZ = 0, DMRGX_OP_SP = 1, DMRGX_OP_EYE = 2, DMRGX_OP_H = 3 };

const char* dmrgx_last_error(void);
/* number of kernels this library has launched so far in this process */
dmrgx_int dmrgx_launch_count(void);

/* ---- context: one CUDA device + stream (replaces the MPI communicator of the reference objects) ---- */
/* stream: a cudaStream_t to run on (e.g. torch's current stream), or NULL to create a private one */
int dmrgx_ctx_create(int device, void* stream, dmrgx_ctx* out);
/* Multi-GPU: one process per GPU.  Rank 0 obtains a 128-byte communicator id (an ncclUniqueId) and the launcher hands it
   to the other ranks (torch.distributed broadcast in bench.py, a file in the driver); every rank then creates its context
   with its rank.  This replaces the MPI communicator the reference objects are created on (MPI_Comm_rank/size,
   include/DMRGBlockContainer.hpp:279-280).  Objects created on such a context are sharded by superblock row ranges:
   the successor of KronSumShellSplitOwnership (src/DMRGKron.cpp:1519-1704). */
int dmrgx_dist_unique_id(void* out128);
int dmrgx_ctx_create_dist(int device, void* stream, int rank, int world, const void* id128, dmrgx_ctx* out);
int dmrgx_ctx_rank(dmrgx_ctx ctx, int* rank, int* world);
int dmrgx_ctx_destroy(dmrgx_ctx ctx);
int dmrgx_ctx_sync(dmrgx_ctx ctx);
/* fill fraction above which a sector-block panel is stored dense (default 0.125) */
int dmrgx_ctx_set_dense_threshold(dmrgx_ctx ctx, double fill);

/* ---- Block::SpinBase (include/DMRGBlock.hpp:79-434) ---- */
/* Initialize(comm, nsites, qn_list, qn_size): include/DMRGBlock.hpp:243-250, src/DMRGBlock.cpp:173-196 */
int dmrgx_block_create(dmrgx_ctx ctx, dmrgx_int nsites, dmrgx_int nsectors, const double* qn_list, const dmrgx_int* qn_size,
                       dmrgx_block* out);
/* Initialize(comm, 1, PETSC_DEFAULT): one site with the default spin operators, src/DMRGBlock.cpp:123-137, 1106-1225.
   spin_twice: 1 = spin-1/2 (default), 2 = spin-1 (-spin option, src/DMRGBlock.cpp:54-94) */
int dmrgx_block_single_site(dmrgx_ctx ctx, int spin_twice, dmrgx_block* out);
/* Sz(i) / Sp(i) / H as CSR with global column indices (what MatGetRow / MatSeqAIJGetArray give).  op in
   {DMRGX_OP_SZ, DMRGX_OP_SP, DMRGX_OP_H}; Sm is derived (CreateSm, src/DMRGBlock.cpp:623-636).  Entries
   outside the operator's sector block fail with 63 like MatCheckOperatorBlocks (src/DMRGBlock.cpp:508-600). */
int dmrgx_block_set_operator(dmrgx_block blk, int op, dmrgx_int isite, const dmrgx_int* rowptr, const dmrgx_int* colidx,
                             const double* values);
/* read an operator back as CSR: call with colidx == NULL to get nnz, then with buffers (rowptr: nstates+1) */
int dmrgx_block_get_operator(dmrgx_block blk, int op, dmrgx_int isite, dmrgx_int* nnz, dmrgx_int* rowptr, dmrgx_int* colidx,
                             double* values);
int dmrgx_block_info(dmrgx_block blk, dmrgx_int* nsites, dmrgx_int* nstates, dmrgx_int* nsectors);
/* Magnetization.List() / Sizes(): include/QuantumNumbers.hpp:84-98 */
int dmrgx_block_sectors(dmrgx_block blk, double* qn_list, dmrgx_int* qn_size);
/* CheckOperatorBlocks: src/DMRGBlock.cpp:603-620 */
int dmrgx_block_check(dmrgx_block blk);
int dmrgx_block_destroy(dmrgx_block blk);
/* KronEye_Explicit(Left, Right, Terms, BlockOut): src/DMRGKron.cpp:459-615.  A right block with one state per sector (a single
   site: the only way the reference's DMRG loop calls it) is enlarged on the device without moving operator data; a general
   right block (several sites / wider sectors, e.g. the reference's TestKron01 case) is assembled from the CSR forms. */
int dmrgx_block_enlarge(dmrgx_block left, dmrgx_block site, dmrgx_int nterms, const double* a, const int* iop, const dmrgx_int* isite,
                        const int* jop, const dmrgx_int* jsite, dmrgx_block* out);

/* ---- KronBlocks_t (include/DMRGKron.hpp:117-480) ---- */
/* ctor :124-213; nqn == 0 keeps every sector (and sorts by descending QN), else only the listed ones */
int dmrgx_kron_create(dmrgx_block left, dmrgx_block right, dmrgx_int nqn, const double* qn_sectors, dmrgx_kron* out);
int dmrgx_kron_destroy(dmrgx_kron k);
dmrgx_int dmrgx_kron_size(dmrgx_kron k);                                 /* size()       :216 */
dmrgx_int dmrgx_kron_num_states(dmrgx_kron k);                           /* NumStates()  :297 */
/* data(): QN, LeftIdx, RightIdx, Sizes (size() entries each) and Offsets (size()+1)  :219-262 */
int dmrgx_kron_data(dmrgx_kron k, double* qn, dmrgx_int* left_idx, dmrgx_int* right_idx, dmrgx_int* sizes, dmrgx_int* offsets);
dmrgx_int dmrgx_kron_map(dmrgx_kron k, dmrgx_int lidx, dmrgx_int ridx);      /* Map(l,r), -1 if absent      :283-294 */
dmrgx_int dmrgx_kron_offsets_lr(dmrgx_kron k, dmrgx_int lidx, dmrgx_int ridx); /* Offsets(l,r), -1 if absent :272-276 */

/* ---- the shell Hamiltonian ---- */
/* KronSumConstruct(Terms, H) with do_shell: src/DMRGKron.cpp:759-841, 1871-1917.  Terms are the full list
   Ham.H(nsites_total); intra-block terms are ignored and the right sites reflected exactly as :788-807. */
int dmrgx_hshell_create(dmrgx_kron k, dmrgx_int nterms, const double* a, const int* iop, const dmrgx_int* isite, const int* jop,
                        const dmrgx_int* jsite, dmrgx_hshell* out);
/* KronConstruct(Mat_L, OpType_L, Mat_R, OpType_R, MatOut): include/DMRGKron.hpp:309 — one term 1.0·A⊗B; an op of
   DMRGX_OP_EYE means identity on that side */
int dmrgx_hshell_create_single(dmrgx_kron k, int op_left, dmrgx_int isite_left, int op_right, dmrgx_int isite_right, dmrgx_hshell* out);
/* correlator operator 1.0 · (O_1·…·O_nl on the left block) ⊗ (O'_1·…·O'_nr on the right block): CalculateOperatorProducts
   (MatMatMult chain in list order) + KronConstruct, include/DMRGBlockContainer.hpp:2262-2296, 2340-2425.  An empty
   list is the identity; ops are DMRGX_OP_SM / SZ / SP, sites are block-local. */
int dmrgx_hshell_create_product(dmrgx_kron k, dmrgx_int nl, const int* lop, const dmrgx_int* lsite, dmrgx_int nr, const int* rop,
                                const dmrgx_int* rsite, dmrgx_hshell* out);
/* MatMult_KronSumShell(A, x, y): src/DMRGKron.cpp:1827-1869.  Device pointers, length NumStates(). */
int dmrgx_hshell_apply(dmrgx_hshell h, const double* d_x, double* d_y);
/* The distributed form of the same callback.  d_x: full-length device buffer in which this rank's rows are valid on entry;
   the VecScatter-to-all of src/DMRGKron.cpp:1833-1834 becomes an in-place sector-halo exchange over NCCL (only the sector pairs
   this rank's rows couple to arrive; the rest of d_x is left as it was), then this rank's rows of d_y (also a full-length
   buffer) are computed.  On one GPU identical to dmrgx_hshell_apply. */
int dmrgx_hshell_apply_sharded(dmrgx_hshell h, double* d_x, double* d_y);
/* bytes of psi this rank RECEIVES per sharded apply (the sector halo: only the X_q panels its tiles read) and what the reference's
   VecScatter-to-all (src/DMRGKron.cpp:1833-1834) would bring it */
int dmrgx_hshell_halo_bytes(dmrgx_hshell h, double* halo_recv_bytes, double* allgather_recv_bytes);
/* rows [begin,end) this rank owns; cuts (optional, world+1 entries) = the ownership table of all ranks */
int dmrgx_hshell_row_range(dmrgx_hshell h, dmrgx_int* begin, dmrgx_int* end, dmrgx_int* cuts);
/* profiling aids: run only stage 1 (V = A·X panels) or stage 2 (Y = Σ V·Bᵀ) of an apply, and their useful flops */
int dmrgx_hshell_apply_stage(dmrgx_hshell h, int stage, const double* d_x, double* d_y);
int dmrgx_hshell_stage_flops(dmrgx_hshell h, double* flops_stage1, double* flops_stage2);
/* the FP64 tensor flops the two launches execute for them (tiles padded to whole DMMA fragments and K chunks) */
int dmrgx_hshell_stage_exec_flops(dmrgx_hshell h, double* flops_stage1, double* flops_stage2);
/* plan introspection: executions per segment type {GEMM, AXPY, DIAG, CSRA, CSRB, CSRADD} over the items of a stage */
int dmrgx_hshell_plan_segtypes(dmrgx_hshell h, int stage, dmrgx_int* out6);
/* plan introspection: per work item {tm, tn, segments, sum of K of its GEMM segments}; returns the item count */
dmrgx_int dmrgx_hshell_plan_items(dmrgx_hshell h, int stage, dmrgx_int cap, dmrgx_int* out4);
/* same with HOST buffers (the Vec arrays of the PETSc callback): H2D, (all-gather,) apply, D2H, synchronous.  x and y are
   this rank's LOCAL rows, as VecGetArray returns them on the reference's MPI vectors — the whole vector on one GPU. */
int dmrgx_hshell_apply_host(dmrgx_hshell h, const double* x, double* y);
/* MatDestroy_KronSumShell: src/DMRGKron.cpp:1919-1942 */
int dmrgx_hshell_destroy(dmrgx_hshell h);
/* algorithmic bytes / flops of one apply (SURVEY.md §8d) and the number of shell terms */
int dmrgx_hshell_stats(dmrgx_hshell h, dmrgx_int* nstates, dmrgx_int* nterms, double* alg_bytes, double* alg_flops,
                       dmrgx_int* ntiles_stage1, dmrgx_int* ntiles_stage2);

/* bytes of device memory one apply streams through besides the original operator panels (V workspace, pre-summed factors, psi, y) */
int dmrgx_hshell_workspace_bytes(dmrgx_hshell h, double* bytes);
/* the algorithmic bytes / flops of the WHOLE operator on a multi-GPU context (dmrgx_hshell_stats then reports this rank's share) */
int dmrgx_hshell_stats_global(dmrgx_hshell h, double* alg_bytes, double* alg_flops);

/* ---- ground state: EPSSolve + EPSGetEigenpair(0), include/DMRGBlockContainer.hpp:1484-1500 ---- */
typedef struct {
    double tol;               /* -H_eps_tol    (SLEPc default 1e-8)  */
    dmrgx_int ncv;            /* -H_eps_ncv    (SLEPc default 16)    */
    dmrgx_int max_it;         /* -H_eps_max_it (0: max(100, 2N/ncv)) */
    unsigned long long seed;  /* start vector */
} dmrgx_eigs_opts;
typedef struct { dmrgx_int nmatvec, nrestart, converged; double resid; } dmrgx_eigs_stats;
int dmrgx_eigs_smallest(dmrgx_hshell h, const dmrgx_eigs_opts* opts, double* e0, double* d_psi, dmrgx_eigs_stats* stats);
/* EXTENSION (no reference counterpart: EPSSolve is never given an initial space there).  The same solve started from
   d_initial (device, global length; on several GPUs every rank passes the whole vector) — the seeded random vector is used
   when d_initial is NULL, zero or not finite.  Same eigenpair to `tol`, fewer H*psi when the guess is good.  A guess with no
   component along the ground state (an exact eigenvector of a block of H, or any vector of an exactly invariant subspace
   without it, such as a symmetry sector) makes the Krylov space break down (||r|| < 1e-14) before the basis is full; the
   solve then goes on from a fresh seeded random direction orthogonal to the basis and does not stop before the end of that
   restart cycle.  It returns the ground state when the steps left in that cycle find a Ritz value below the lowest one of
   the exhausted space (a space of dimension close to ncv leaves too few of them).  A guess whose ground-state component is
   rounding-sized but not zero does not break down: its Krylov space leaves the subspace along that noise, and the result
   depends on it.  An exact ground state as the guess still costs one whole cycle, min(ncv, dimension) H*psi. */
int dmrgx_eigs_smallest_from(dmrgx_hshell h, const dmrgx_eigs_opts* opts, const double* d_initial, double* e0, double* d_psi, dmrgx_eigs_stats* stats);

/* ---- EXTENSION: wave-function transformation (S. R. White, PRL 77, 3633 (1996)) — the guess for dmrgx_eigs_smallest_from.
   The reference has none (include/DMRGBlockContainer.hpp:1484-1500 starts every step from a random vector); the driver uses this
   only under -wavefunction_prediction 1.
     dmrgx_wave_create : after dmrgx_truncate of a step — psi of superblock k with the side that grows in the next step projected
                         on its kept states (grown_side = that side's dmrgx_xform; grow_left != 0: the left block grows).
     dmrgx_wave_apply  : in the next step — shrinking_side = the dmrgx_xform that CREATED the other block of the previous step
                         from the block now in its place, site = the single-site block, k_new = the new superblock.  Writes
                         the guess (global length of k_new) and *ok = 1, or *ok = 0 when the sector structures do not chain up
                         (first step of a sweep, blocks replaced in between): the caller then starts from the random vector. */
typedef struct dmrgx_wave_s* dmrgx_wave;
int dmrgx_wave_create(dmrgx_kron k, const double* d_psi, dmrgx_xform grown_side, int grow_left, dmrgx_wave* out);
int dmrgx_wave_apply(dmrgx_wave w, dmrgx_xform shrinking_side, dmrgx_block site, dmrgx_kron k_new, double* d_psi_new, int* ok);
int dmrgx_wave_destroy(dmrgx_wave w);

/* ---- truncation: GetTruncation, include/DMRGBlockContainer.hpp:1656-1959 ---- */
int dmrgx_truncate(dmrgx_kron k, const double* d_psi, dmrgx_int mstates, dmrgx_xform* left, dmrgx_xform* right);
/* m = RotMatT rows, nstates = columns, nsectors of BT.QN, TruncErr, and the size of the grouped spectrum */
int dmrgx_xform_info(dmrgx_xform x, dmrgx_int* m, dmrgx_int* nstates, dmrgx_int* nsectors, double* trunc_err, dmrgx_int* nspectrum);
int dmrgx_xform_sectors(dmrgx_xform x, double* qn_list, dmrgx_int* qn_size);
/* unsorted, grouped eigenvalues + their block index, as SaveEntanglementSpectra dumps them (:1790-1793) */
int dmrgx_xform_spectrum(dmrgx_xform x, double* eigval, dmrgx_int* blk_idx);
/* RotMatT as a dense m × nstates row-major host matrix (debug / parity) */
int dmrgx_xform_rotmat(dmrgx_xform x, double* out);
int dmrgx_xform_destroy(dmrgx_xform x);

/* ---- rotation: SysBlockOut.Initialize(nsites, BT.QN) + RotateOperators(SysBlockEnl, RotMatT),
        include/DMRGBlockContainer.hpp:1561-1563, src/DMRGBlock.cpp:677-823 ---- */
int dmrgx_rotate(dmrgx_block enlarged, dmrgx_xform x, dmrgx_block* out);

/* ---- correlator kernel: <psi| A⊗B |psi> = VecDot(psi, MatMult(H1, psi)), include/DMRGBlockContainer.hpp:2287-2296 ---- */
int dmrgx_expect(dmrgx_hshell h1, const double* d_psi, double* value);

/* ---- EXTENSION: the all-pairs spin correlation matrix (no reference counterpart: there every correlator is one
   KronConstruct + MatMult + VecDot, include/DMRGBlockContainer.hpp:2262-2296).  For the n = nL + nR superblock sites
   (site s < nL is left-block site s, site s >= nL is right-block site nL+nR-1-s, as in dmrgx_hshell_create) and psi in the
   superblock's one total-Sz sector, used as given (not normalised):
       szsz[i*n+j] = <psi| Sz_i Sz_j |psi>,  spsm[i*n+j] = <psi| S+_i S-_j |psi>,  smsp[i*n+j] = <psi| S-_i S+_j |psi>,
       sz[i] = <psi| Sz_i |psi>
   all host buffers (n×n row-major, n).  One batched device pass: per operator type the panels O_s·psi of every site are
   built by one contraction launch and reduced to their Gram matrix by one FP64 tensor-core launch; the same-block entries
   equal the operator products of dmrgx_hshell_create_product.  flops (may be NULL) receives the algorithmic flops of the
   call.  On a multi-GPU context the calling rank computes everything from its complete psi, with no collective.
   Errors: 62 psi or an output NULL, 56 the kron has not exactly one sector, 73 a block lacks Sz_i or Sp_i (site in the message). */
int dmrgx_corr_matrix(dmrgx_kron k, const double* d_psi, double* szsz, double* spsm, double* smsp, double* sz, double* flops);

/* ---- EXTENSION: the dimer (bond–bond) correlation matrix (no reference counterpart: there every four-operator correlator
   would be nine KronConstruct + MatMult + VecDot, include/DMRGBlockContainer.hpp:2262-2296).  Bond a joins the superblock
   sites site_i[a] != site_j[a] (numbered as in dmrgx_corr_matrix) and stands for the isotropic bond operator, in this order:
       D_a = Sz_i Sz_j + ½ S+_i S-_j + ½ S-_i S+_j
   psi lies in the superblock's one total-Sz sector and is used as given (not normalised).  Host outputs:
       dd[a*nbonds+b] = <D_a psi, D_b psi> = <psi| D_aᵀ D_b |psi>   (nbonds×nbonds row-major),   d[a] = <psi| D_a |psi>
   Ordering convention: every operator is its block's stored (rotated) matrix, so on a truncated block two operators of the
   same block do not commute; a same-block bond is the product in the order above and its adjoint is
   D_aᵀ = Sz_j Sz_i + ½ S+_j S-_i + ½ S-_j S+_i.  Then d[a] = szsz + ½(spsm + smsp) at [i*n+j] of dmrgx_corr_matrix to rounding,
   and on exact blocks dd is the true <(S_i·S_j)(S_k·S_l)>.  Nothing is symmetrised.
   One batched device pass: the panels O_j·psi (O in Sz, S-, S+) of the bonds' second sites, then every bond panel D_a·psi
   (one contraction launch each), then one Gram matrix over the bond panels and psi.  Device memory during the call:
   (nj·(D + D₋ + D₊) + (nbonds + 1)·D)·8 bytes plus the plans, with D the superblock dimension, D∓ those of the sectors qn ∓ 1
   and nj <= n the number of distinct second sites; an empty qn ± 1 sector drops its term.  flops (may be NULL) receives the
   algorithmic flops of the call.  On a multi-GPU context the calling rank computes everything from its complete psi, with
   no collective.
   Errors: 62 psi, a site array or an output NULL; 63 nbonds < 1, or a site outside [0, n) or site_i == site_j (the bond
   index in the message); 56 the kron has not exactly one sector; 73 a block lacks Sz or Sp at a site of some bond (site in
   the message). */
int dmrgx_dimer_matrix(dmrgx_kron k, const double* d_psi, dmrgx_int nbonds, const dmrgx_int* site_i, const dmrgx_int* site_j, double* dd,
                       double* d, double* flops);

/* ---- EXTENSION: the dynamical structure factor by the continued-fraction method (K. Hallberg, PRB 52, R9827 (1995); no reference
   counterpart).  psi lies in the one total-Sz sector qn of k and is used as given (not normalised); op is DMRGX_OP_SZ, DMRGX_OP_SP
   or DMRGX_OP_SM, whose value is the sector shift.  Vector v (v < nvec) starts from
       phi_v = Σ_s coef[v*n+s] · O_s psi      (O = Sz, S+ or S-, superblock sites s < n numbered as in dmrgx_corr_matrix)
   in the sector qn + op, and h_target is a shell on a kron of the SAME two block objects whose single sector is qn + op (for
   DMRGX_OP_SZ the step's own Hamiltonian).  From phi_v/‖phi_v‖ a plain three-term Lanczos recurrence of h_target runs, with no
   reorthogonalisation; its coefficients give  G_v(z) = <phi_v| (z - H)^-1 |phi_v> = norm2[v] / (z - α_0 - β_1²/(z - α_1 - …))
   and reproduce the moments <phi_v| H^k |phi_v> for k < 2·nsteps.  Host outputs:
       alpha[v*nsteps+t] = α_t,  beta[v*nsteps+t] = β_t (the coupling of steps t-1 and t, β_0 = 0),  norm2[v] = <phi_v, phi_v>,
       nsteps_done[v] <= nsteps: the recurrence stops at an invariant subspace, β_{t+1} <= 1e-10·sqrt(α_t² + β_t²); later
       entries are 0.  A start vector with ‖phi_v‖ <= 1e-12 · Σ_s |coef_s|·‖O_s psi‖ is zero up to rounding: norm2 = 0, no steps.
   One batched device pass: the n panels O_s psi are one contraction launch, the start vectors of a batch are one GEMM over
   them, and a batch of nb vectors keeps three columns each on the device (v_prev, v, H·v; nb = 2 GiB / (24·D), at least 1,
   D the dimension of the sector qn + op).  Every step applies h_target once per vector and advances the whole batch with two
   launches, with no host synchronisation until the batch is done.  Device memory during the call: (n + 3·nb)·D·8 bytes plus
   the plans.  Each vector's sums run in a fixed order that does not depend on nb: a vector gives the same bits alone or in a
   batch.  flops (may be NULL) receives the algorithmic flops: panels + start vectors + nvec·nsteps applies + recurrence.
   Errors: 62 psi, h_target, coef or an output NULL; 63 op not one of the three, nvec < 1, nsteps < 1 or a coefficient not
   finite; 56 k has not exactly one sector, or the context is multi-GPU (the sharded apply is collective); 73 h_target is not
   on the sector qn + op of the same blocks, or a block lacks Sz or Sp at a site with a non-zero coefficient (site in the
   message). */
int dmrgx_spectral_lanczos(dmrgx_kron k, const double* d_psi, dmrgx_hshell h_target, int op, dmrgx_int nvec, const double* coef,
                           dmrgx_int nsteps, double* alpha, double* beta, double* norm2, dmrgx_int* nsteps_done, double* flops);

/* ---- EXTENSION: the real-space dynamical correlation matrix (no reference counterpart).  dmrgx_spectral_lanczos, which it calls
   with the same contract, bits and error codes for alpha, beta, norm2 and nsteps_done, plus at every step the overlap of each
   normalised Lanczos vector v_t of vector v (v_0 = phi_v/‖phi_v‖) with all n single-site panels:
       overlaps[(v*nsteps + t)*n + s] = <O_s psi, v_t>      t < nsteps_done[v];  0 for t >= nsteps_done[v].
   With T_v the tridiagonal matrix of α and β and k < nsteps_done[v], the three-term relation H·V = V·T + β·v·eᵀ, which holds to
   rounding however much orthogonality is lost, gives the mixed moments exactly
       <O_s psi| H^k |phi_v> = ‖phi_v‖ Σ_t overlaps[v][t][s] · (T_v^k)_{t,0},
   and in the same way  <O_s psi| (z - H)^-1 |phi_v> ≈ ‖phi_v‖ Σ_t ov·[(z - T_v)^-1]_{t,0}  and
   <O_s psi| e^{-i(H - E0)τ} |phi_v> ≈ ‖phi_v‖ Σ_t ov·[e^{-i(T_v - E0)τ}]_{t,0}.  At equal time √norm2[v]·ov[v][0][s] =
   <O_s psi, phi_v> (the coef-weighted row of SzSz, SpSm or SmSp of dmrgx_corr_matrix for op Sz, S- or S+) and
   Σ_s coef[v][s]·ov[v][0][s] = √norm2[v].  With coef rows e_c, vector v gives the column c of <O_s psi| f(H) |O_c psi> for
   every s and any f.  Every site's panel is built, so every site needs Sz and Sp (73 otherwise).  Each step adds one
   rectangular Gram launch pair over the n panels and the batch's vectors; each element's sums run in a fixed order that
   depends only on its two columns and D, so a vector's overlaps are the same bits alone or in a batch.  Device memory:
   (n + 3·nb)·D·8 bytes, plus nb·nsteps·n·8 bytes of overlaps, plus the Gram slab partials (⌈D/8192⌉·⌈n/32⌉·⌈nb/32⌉·8 KiB)
   and the plans.  flops adds 2·n·D per vector and step.  Errors: those of dmrgx_spectral_lanczos, and 62 overlaps NULL. */
int dmrgx_spectral_lanczos_overlaps(dmrgx_kron k, const double* d_psi, dmrgx_hshell h_target, int op, dmrgx_int nvec, const double* coef,
                                    dmrgx_int nsteps, double* alpha, double* beta, double* norm2, dmrgx_int* nsteps_done, double* overlaps,
                                    double* flops);

/* ---- Hamiltonians::J1J2XXZModel_SquareLattice::H(nsites): src/Hamiltonians.cpp:73-122 (host only).
        Returns the number of terms (fills at most maxterms); bc: 0 open, 1 periodic; nsites < 0 = full lattice. ---- */
dmrgx_int dmrgx_ham_terms(dmrgx_int Lx, dmrgx_int Ly, double J1, double Jz1, double J2, double Jz2, int bcx, int bcy, dmrgx_int nsites,
                          dmrgx_int maxterms, double* a, int* iop, dmrgx_int* isite, int* jop, dmrgx_int* jsite);

/* ---- microbenchmark of the contraction engine on one plain product C[M,N] = Σ_seg A_seg·B_segᵀ (operand layouts selectable),
        used by tools/ and the profiles; not part of the reference's surface ---- */
int dmrgx_selftest_gemm(dmrgx_ctx ctx, dmrgx_int M, dmrgx_int N, dmrgx_int K, int a_k_contig, int b_k_contig, int nseg, int reps, double* ms,
                        double* max_err);

/* ---- the batched symmetric eigensolver of the truncation (EigRDM_BlockDiag, include/DMRGBlockContainer.hpp:1962-2003) on caller-supplied
        matrices: nblocks row-major symmetric matrices of orders n[b], concatenated in `a` (host).  On return `a` holds the eigenvectors (row k of
        block b = k-th eigenvector, ascending eigenvalues) and `w` (sum of n[b] entries) the eigenvalues; *ms = device time of the solve.
        A test / profiling aid, not part of the reference's surface. ---- */
int dmrgx_selftest_eig(dmrgx_ctx ctx, dmrgx_int nblocks, const dmrgx_int* n, double* a, double* w, double* ms);

/* ---- device vectors (the Vec objects of the callers) ---- */
int dmrgx_vec_alloc(dmrgx_ctx ctx, dmrgx_int n, double** d_out);
int dmrgx_vec_free(dmrgx_ctx ctx, double* d);
int dmrgx_vec_set(dmrgx_ctx ctx, double* d_dst, const double* h_src, dmrgx_int n);
int dmrgx_vec_get(dmrgx_ctx ctx, double* h_dst, const double* d_src, dmrgx_int n);

#ifdef __cplusplus
}
#endif
#endif /* DMRGX_H */
