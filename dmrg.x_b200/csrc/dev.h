/*  dev.h — the thin device layer.  Everything above it (block.cpp, hshell.cpp, eigs.cpp, truncate.cpp,
 *  predict.cpp, plan.cpp, abi.cpp) is plain C++ that plans work on the host and hands flat POD work lists
 *  to the sm_100a kernels in dev_cuda.cu through the functions declared here.
 *
 *  The product library libdmrgx_b200.so links dev_cuda.cu and nothing else behind this interface; there
 *  is no CPU implementation in the product.  (tests/plancheck/dev_host.cpp re-implements this header
 *  with naive host loops ONLY so that `pytest -m "not gpu"` can check the host-side planning logic —
 *  offsets, strides, sector maps — in a container without a GPU; it is never part of the product.)
 */
#pragma once
#include <cstddef>
#include <cstdint>

namespace dev {

/* ------------------------------------------------------------------------------------------------
 *  The one compute engine: every contraction of the hot path is a list of output tiles ("work
 *  items"), each accumulating a chain of segments in registers and writing its tile exactly once.
 *      GEMM  : acc(m,n) += coef * Σ_k A(m,k) · B(k,n)      A(m,k)=A[m*lda_m+k*lda_k], B(k,n)=B[n*ldb_n+k*ldb_k]
 *      AXPY  : acc(m,n) += coef * A(m,n)                    (n uses lda_k as its stride)
 *      DIAG  : acc(m,n) += coef * [m + drow == n]
 *      CSRA  : acc(m,n) += coef * Σ_{e in row (row0+m)} val[e] · B(colidx[e], n)      (sparse left factor)
 *      CSRB  : acc(m,n) += coef * Σ_{e in row (row0+n)} val[e] · A(m, colidx[e])      (sparse right factor)
 *      CSRADD: acc(m,n) += coef * Σ_{e in row (row0+m)} val[e] · [colidx[e] == n + dcol]
 *  Fast (FP64 DMMA) GEMM layouts: lda_k==1 or lda_m==1, and ldb_k==1 or ldb_n==1.
 *  Pointer fields of the sparse segments: B = CSR values; A = the dense operand — for CSRA the right
 *  factor addressed with (ldb_k, ldb_n), for CSRB the left factor addressed with (lda_m, lda_k).
 * ---------------------------------------------------------------------------------------------- */
enum SegType : int { SEG_GEMM = 0, SEG_AXPY = 1, SEG_DIAG = 2, SEG_CSRA = 3, SEG_CSRB = 4, SEG_CSRADD = 5 };

struct Segment {
    const double* A;
    const double* B;      /* CSR*: values */
    const int* rowptr;    /* CSR* */
    const int* colidx;    /* CSR*: indices local to the tile the CSR block describes */
    long long lda_m, lda_k;
    long long ldb_n, ldb_k;
    double coef;
    int K;
    int type;
    int row0;             /* CSR row that corresponds to row 0 (CSRA/CSRADD) or column 0 (CSRB) of the cell */
    int d;                /* DIAG: drow; CSRADD: dcol */
    int flags;            /* SEGF_A_X / SEGF_B_X: the pointer field holds a BYTE OFFSET into the x vector of the launch */
    int pad;
};
enum : int { SEGF_A_X = 1, SEGF_B_X = 2 };

struct WorkItem {
    double* C;            /* tile origin */
    long long ldc;
    int m0, n0;           /* origin of the tile inside its cell: operand bases are A + m0*lda_m, B + n0*ldb_n */
    int tm, tn;           /* extents, 1..TILE */
    int seg_begin, seg_end;
    int mode;             /* 0: store (C = acc), 1: atomic accumulate (C += acc) */
    int c_in_y;           /* 0: C is a pointer; 1: C holds a BYTE OFFSET into the y vector of the launch; 2: into the w scratch */
};

constexpr int TILE = 64;  /* maximum tile extent of a work item */

struct Stream;            /* device, stream, device heap, communicator */

int init(int device, void* user_stream, Stream** out); /* 0 on success; fails loudly without a CUDA device */
void destroy(Stream*);
const char* last_error();
void make_current(Stream*);   /* cudaSetDevice(device of the stream): called at every C-ABI entry point */

void* malloc_bytes(Stream*, size_t bytes);
void free_bytes(Stream*, void* p);
void h2d(Stream*, void* dst, const void* src, size_t bytes);
void d2h(Stream*, void* dst, const void* src, size_t bytes);
void d2d(Stream*, void* dst, const void* src, size_t bytes);
void memset0(Stream*, void* dst, size_t bytes);
void sync(Stream*);
/* number of kernel launches issued through this layer so far (bench.py's gpu_launches) */
long long launch_count();

/* ---- collectives: one process per GPU, NCCL over NVLink/NVSwitch (SURVEY.md §8e).  The exchange steps of the path: the
   sector-halo exchange of the sharded superblock vector before an apply, the all-reduce of a handful of scalars per
   Lanczos step, in-place all-gathers of the finished ground state and of the rotated-operator panels, and broadcasts of
   density-matrix eigenvectors and eigenvalues from the rank that computed them.  All calls are enqueued on the context's
   stream (device-ordered, no host synchronisation). ---- */
constexpr int COMM_ID_BYTES = 128;                       /* ncclUniqueId */
int comm_unique_id(void* out);                           /* rank 0 creates it, the launcher hands it to the others */
int comm_init(Stream*, int rank, int world, const void* id);
void allreduce_sum(Stream*, double* d_buf, long long n); /* in place */
/* in place: rank r owns d_buf[offsets[r] .. offsets[r+1]) and receives all other ranges */
void allgatherv(Stream*, double* d_buf, const long long* offsets);
/* sector-halo exchange: transfer i moves d_buf[off[i] .. off[i]+cnt[i]) from rank from[i] to rank to[i] (same place in the
   receiver's buffer); the same list on every rank, one NCCL group of point-to-point transfers */
void exchange_ranges(Stream*, double* d_buf, int n, const int* from, const int* to, const long long* off, const long long* cnt);
/* a batch of broadcasts, root[i] sends d_ptr[i][0..count[i]) to everybody (one NCCL group) */
void bcast_batch(Stream*, int n, double* const* d_ptr, const long long* count, const int* root);

/* chain contraction engine */
/* x / y: base pointers that offset-typed operands (SEGF_*_X, c_in_y) are relative to, so one plan serves any
   pair of device vectors (the Lanczos basis vectors change every step; the plan does not). */
void run_chain(Stream*, const WorkItem* d_items, int nitems, const Segment* d_segs, const double* x, double* y, double* w = nullptr);

/* ------------------------------------------------------------------------------------------------
 *  Sparse-sector SpMM (north_star (a)): Y_p = Σ_t coef_t · A_t[IL,JL] · X_q(t) · B_t[IR,JR]ᵀ with every factor a sparse matrix
 *  (or the identity), all terms of a sector pair fused: one CTA per (pair, 8 consecutive left rows), threads along the right
 *  index with all 8 rows of their columns in registers; the CTA's own rows of X_p are staged in shared memory by one TMA bulk
 *  copy; y is written exactly once.  At plan time the terms and the left factors are flattened into ROW PROGRAMS: short
 *  lists of (source row of psi, weight[, right factor]) entries, so that the CTA reaches its psi loads after two dependent
 *  fetches and has the loads of eight rows in flight together.
 * ---------------------------------------------------------------------------------------------- */
constexpr int SP_ROWS = 4;          /* left rows per CTA */
/* Row programs, slot-major: slot k holds the k-th entry of EACH of the tile's 8 rows, so that a CTA issues the psi loads of
   eight rows at once.  src = element offset in x of the source row of X_q; rows with fewer entries carry w = 0 and a valid src. */
struct SpASlot { long long src[SP_ROWS]; double w[SP_ROWS]; };   /* identity on the right, source row in L2: acc(r,c) += w_r · x[src_r + c] */
struct SpSSlot { int roff[SP_ROWS]; int pad[SP_ROWS]; double w[SP_ROWS]; }; /* the same with the source row inside the tile: acc(r,c) += w_r · xs[roff_r + c] */
/* a right factor B: acc(r,c) += w_r · Σ_t eval[t*ld + c] · X_r[ecol[t*ld + c]], t < W (ELL, slot-major over the output
   columns: coalesced reads; padding = value 0, column 0).  X_r = xs + roff[r] when all_in (every source row is one of the tile's
   own: decided at plan time, no generic pointers in the kernel), else x + src[r]. */
struct SpBSlot { const int* ecol; const double* eval; int W, ld; int all_in, pad; int roff[SP_ROWS]; long long src[SP_ROWS]; double w[SP_ROWS]; };
struct SpTile {
    long long off;                  /* element offset in x and y of the tile's first row */
    int nR, nrows;
    int a_begin, a_count;           /* SpASlot records of the tile */
    int s_begin, s_count;           /* SpSSlot records */
    int b_begin, b_count;           /* SpBSlot records */
    int pad[6];
};
constexpr int SP_MAX_NR = 3072;     /* widest right sector the kernel stages (8 rows x 3072 doubles = 192 KB of shared memory) */
void run_spmm(Stream*, const SpTile* d_tiles, int ntiles, const SpASlot* d_aslots, const SpSSlot* d_sslots, const SpBSlot* d_bslots, const double* x, double* y,
              int max_nR);

/* Long accumulation chains are cut into parts that write partial tiles to the w scratch (so that a launch has enough
   equal work items to fill 148 SMs several times over); the parts are then summed in a FIXED order — deterministic,
   no atomics.  dst: byte offset into y (dst_in_y) or pointer; part p of the tile is the row-major tm×tn panel at
   w + src_off/8 + p*tm*tn. */
struct ReduceItem {
    double* dst;
    long long ldc;
    long long src_off;   /* bytes into w */
    int tm, tn;
    int nparts;
    int dst_in_y;
};
void run_reduce(Stream*, const ReduceItem* d_items, int nitems, double* y, const double* w);

/* vector kernels of the thick-restart Lanczos (all results stay on the device) */
/* x[i] = u(seed, first + i): depends on the GLOBAL index only */
void fill_random(Stream*, double* x, long long n, unsigned long long seed, long long first = 0);
/* One fused Gram-Schmidt pass over the basis (a single read of V, deterministic reductions finished by the last block, no
   host involvement):   if d_coef:  w -= Σ_i d_coef[i]·V_i   (in place);   then, on the updated w,
   if d_dots: d_dots[i] = V_i·w (i < nvec);   if d_nrm2: *d_nrm2 = w·w.   nvec <= MAX_BASIS. */
constexpr int MAX_BASIS = 39; /* largest ncv the fused kernels take (eigs_smallest validates -H_eps_ncv against it) */
void gs_pass(Stream*, const double* V, long long ldv, int nvec, double* w, long long n, const double* d_coef, double* d_dots, double* d_nrm2);
/* Last step of the two-pass Gram-Schmidt, fused with the normalisation (no reduction, no all-reduce):
       vout = (w - Σ_i d_coef[i]·V_i) / sqrt(b2),   b2 = *d_nrm2_in - Σ_i d_coef[i]²   (Pythagoras: d_nrm2_in is ||w||² BEFORE the update
   and the coefficients of a second pass are round-off sized, so there is no cancellation);  *d_nrm2_out = b2.  nvec <= MAX_BASIS + 1.
   Refinement "if needed" (what SLEPc's default orthogonalisation does with a much looser test): when Σ_i d_coef[i]² <=
   GS_REFINE_REL² · *d_nrm2_in the correction is not applied — vout = w / sqrt(*d_nrm2_in), b2 = *d_nrm2_in — and V is not read. */
constexpr double GS_REFINE_REL = 1e-12;
void gs_final(Stream*, const double* V, long long ldv, int nvec, const double* w, long long n, const double* d_coef, const double* d_nrm2_in,
              double* d_nrm2_out, double* vout);
/* v = w / sqrt(*d_nrm2) */
void scale_inv_norm(Stream*, const double* w, const double* d_nrm2, double* v, long long n);
/* in place: V_a <- Σ_i S[i*kk+a] V_i  (i < ncv, a < kk), S on the device */
void ritz_rotate(Stream*, double* V, long long ldv, long long n, int ncv, const double* d_S, int kk);
/* *d_out = x·y (the reduction of gs_pass: one launch, fixed summation order) */
void dot(Stream*, const double* x, const double* y, long long n, double* d_out);
/* Gram matrix of a column panel: d_G = PᵀP, row-major np×np and exactly symmetric, over rows [0,n) of the columns
   P + c·ldp (c < np).  P must be 16-byte aligned and ldp even.  FP64 DMMA on the 32×32 tiles on or above the diagonal;
   the rows are cut into fixed slabs whose partial tiles are summed in a fixed order (no atomics: two calls on the same
   data give the same bits), then mirrored.  Two launches. */
void gram(Stream*, const double* P, long long ldp, int np, long long n, double* d_G);
/* Rectangular Gram matrix of two column panels: d_G[i·gs + j·gc] = Σ_{r<n} P[i][r]·Q[j][r] for i < np, j < nq, columns
   P + i·ldp and Q + j·ldq (gram's alignment preconditions for both).  gram's tiles, slabs and fixed slab order, every tile
   computed; the bits of G[i][j] depend only on column i of P, column j of Q and n, never on np, nq or the tile that holds
   them.  n <= 0 writes zeros.  Two launches. */
void gram_rect(Stream*, const double* P, long long ldp, int np, const double* Q, long long ldq, int nq, long long n, double* d_G, long long gs,
               long long gc);

/* Plain three-term Lanczos recurrence over nb independent columns (spectral.cpp), all state on the device.  Column c of a
   slot is slot + c·ld, rows [0, n).  The caller keeps three slots per column and rotates them (prev, cur, y) <- (cur, y, prev)
   after passes 0 and 2; y = H·cur is its own apply.  cur holds u_t = c_t·v_t (c_t = *scale, the norm the recurrence found).
     pass 0 (start):  b2 = y·y;  norm2 = b2, or 0 when b2 <= zero2 (the column is then done with 0 steps), else scale = sqrt(b2)
     pass 1 (step t): cur = v_t = cur / c_t;  y = w = y / c_t - β_t·prev  (β_0 = 0, prev unread);  α_t = v_t·w
                      t = nsteps - 1: the column is done with nsteps steps
     pass 2 (step t): y = w - α_t·v_t;  β_{t+1}² = y·y;  β_{t+1} <= LANCZOS_BETA_REL·sqrt(α_t² + β_t²): done with t + 1 steps,
                      else beta[t+1] = β_{t+1} and scale = β_{t+1}
   A done column is skipped by every later pass.  Each column's sums are cut into lanczos_blocks(n) fixed block partials that
   the column's last block adds in block order: the bits of a column do not depend on nb or on the other columns.  One launch
   per pass for the whole batch. */
constexpr double LANCZOS_BETA_REL = 1e-10;
struct LanczosBatch {
    int nb = 0, nsteps = 0;
    long long n = 0, ld = 0;
    double* alpha = nullptr;        /* nb × nsteps: α_t */
    double* beta = nullptr;         /* nb × nsteps: β_t, β_0 = 0 (zeroed by the caller, like alpha) */
    double* norm2 = nullptr;        /* nb */
    long long* ndone = nullptr;     /* nb, zeroed by the caller */
    double* a = nullptr;            /* nb: α of the current step */
    double* scale = nullptr;        /* nb: c_t */
    const double* zero2 = nullptr;  /* nb */
    int* done = nullptr;            /* nb, zeroed by the caller */
    double* partials = nullptr;     /* nb × lanczos_blocks(n) */
    unsigned int* tickets = nullptr; /* nb, zeroed by the caller; every pass leaves them zero */
};
int lanczos_blocks(long long n);
void lanczos_batch(Stream*, const LanczosBatch&, int pass, int t, const double* prev, double* cur, double* y);

/* dense symmetric eigendecomposition of a batch of independent blocks, in place: block b is n[b]×n[b] at d_A[b]; on exit
   row k of it (row-major) is the k-th eigenvector, eigenvalues ascending in d_w[b].  Blocks of up to 64 states are solved by
   one cyclic-Jacobi launch on a side stream; the larger ones, all together, by batched block Jacobi on the main stream.
   Ordered after everything queued on the main stream, which continues only when all blocks are done.  Returns 0 or the
   first failure. */
int syevd_batch(Stream*, int nblocks, const int* n, double* const* d_A, double* const* d_w);
/* dst[k][:] = src[(n-1-k)][:], k < m   (the m largest eigenvectors, descending) */
void gather_rows_reversed(Stream*, const double* src, int n, int m, double* dst);
/* |x_i| < tol -> 0 */
void filter_small(Stream*, double* x, long long n, double tol);
/* out[i] = a[i] + alpha*b[i] (a may be null -> alpha*b) */
void axpby_out(Stream*, const double* a, const double* b, double alpha, double* out, long long n);

}  // namespace dev
