/*  eigs.cpp — device-resident thick-restart Lanczos replacing the SLEPc call site
 *  include/DMRGBlockContainer.hpp:1484-1500 (EPS_HEP, EPS_SMALLEST_REAL, nev = 1, Krylov-Schur).
 *
 *  The basis (ncv+1 vectors of length D), the work vector and every inner product live in HBM; per
 *  Lanczos step the host sees ncv+2 doubles (the orthogonalisation coefficients and the residual
 *  norm).  Same stopping rule as SLEPc's default: ||r|| <= tol·|theta|, tested at every restart;
 *  same knobs (-H_eps_tol, -H_eps_ncv, -H_eps_max_it).
 */
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "common.h"

namespace dmrgx {

/* tiny dense symmetric eigensolver for the (<= ncv × ncv) projected problem: cyclic Jacobi on the
   host.  Ascending eigenvalues; column k of S (row-major n×n) is eigenvector k. */
static void small_sym_eig(int n, std::vector<double> A, std::vector<double>& w, std::vector<double>& S) {
    S.assign((size_t)n * n, 0.0);
    for (int i = 0; i < n; ++i) S[(size_t)i * n + i] = 1.0;
    auto a = [&](int i, int j) -> double& { return A[(size_t)i * n + j]; };
    for (int sweep = 0; sweep < 100; ++sweep) {
        double off = 0, diag = 0;
        for (int i = 0; i < n; ++i) { diag += a(i, i) * a(i, i); for (int j = i + 1; j < n; ++j) off += a(i, j) * a(i, j); }
        if (off == 0.0 || off <= 1e-34 * (diag + off)) break;
        for (int p = 0; p < n; ++p)
            for (int q = p + 1; q < n; ++q) {
                if (a(p, q) == 0.0) continue;
                const double theta = (a(q, q) - a(p, p)) / (2.0 * a(p, q));
                const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
                const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < n; ++k) { const double x = a(k, p), y = a(k, q); a(k, p) = c * x - s * y; a(k, q) = s * x + c * y; }
                for (int k = 0; k < n; ++k) { const double x = a(p, k), y = a(q, k); a(p, k) = c * x - s * y; a(q, k) = s * x + c * y; }
                for (int k = 0; k < n; ++k) { const double x = S[(size_t)k * n + p], y = S[(size_t)k * n + q]; S[(size_t)k * n + p] = c * x - s * y; S[(size_t)k * n + q] = s * x + c * y; }
            }
    }
    std::vector<int> ord(n);
    for (int i = 0; i < n; ++i) ord[i] = i;
    std::vector<double> d(n);
    for (int i = 0; i < n; ++i) d[i] = a(i, i);
    std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return d[x] < d[y]; });
    std::vector<double> S2((size_t)n * n);
    w.resize(n);
    for (int k = 0; k < n; ++k) { w[k] = d[ord[k]]; for (int i = 0; i < n; ++i) S2[(size_t)i * n + k] = S[(size_t)i * n + ord[k]]; }
    S.swap(S2);
}

double eigs_smallest(HShell* H, const EigsOpts& opts, double* d_psi, EigsStats* stats_out, const double* d_init) {
    Ctx* ctx = H->ctx;
    dev::Stream* st = ctx->st;
    /* Multi-GPU: every rank keeps only its own rows [R0, R0+N) of the Krylov basis; the matvec all-gathers the current
       vector into a full-length buffer and every inner product is completed by an all-reduce of a few doubles.  All
       ranks see identical reduced values, so they take identical decisions without further communication. */
    const long long NG = H->n;                       /* global length */
    const long long R0 = H->row_begin;
    const long long N = H->row_end - H->row_begin;   /* local rows */
    const bool dist = ctx->world > 1;
    EigsStats stats;
    if (NG <= 0) throw Err(ERR_GENERIC, "empty superblock");
    /* the fused Gram-Schmidt and Ritz-rotation kernels keep the whole basis of a cycle in registers: at most 39 vectors */
    if (opts.ncv > dev::MAX_BASIS) throw Err(ERR_ARG_OUTOFRANGE, "-H_eps_ncv is limited to " + std::to_string(dev::MAX_BASIS) + " on this path (got " + std::to_string(opts.ncv) + ")");
    const int ld = (int)std::max<long long>(1, std::min<long long>(opts.ncv < 2 ? 2 : opts.ncv, NG));
    /* SLEPc default max_it = max(100, 2N/ncv) restarts (SURVEY.md Appendix A) */
    const long long max_it = opts.max_it > 0 ? opts.max_it : std::max<long long>(100, 2 * NG / ld);
    BufRef basis = std::make_shared<DevBuf>(ctx, (size_t)(ld + 1) * std::max<long long>(1, N) * 8);
    BufRef wbuf = std::make_shared<DevBuf>(ctx, (size_t)std::max<long long>(1, N) * 8);
    BufRef xfull = dist ? std::make_shared<DevBuf>(ctx, (size_t)NG * 8) : nullptr;
    /* coefficient table: one row per Lanczos step of a restart cycle = {pass-1 coefficients (ld+1), pass-2 coefficients
       (ld+1), ||w'||^2 after the first pass, beta^2 = ||w''||^2}.  It is read back ONCE per cycle: the steps of a cycle are queued
       without any host round trip. */
    const int RW = 2 * (ld + 1) + 2;
    BufRef scal = std::make_shared<DevBuf>(ctx, (size_t)(ld * RW + 2 + ld * ld) * 8);
    double* V = basis->as<double>();
    double* w = wbuf->as<double>();
    double* d_tab = scal->as<double>();
    double* d_nrm2 = d_tab + (size_t)ld * RW;
    double* d_S = d_nrm2 + 2;
    std::vector<double> hh((size_t)ld * RW);
    std::vector<double> T((size_t)ld * ld, 0.0);

    Trace tr(ctx, "eigs");
    bool have_start = false;
    if (d_init) { /* a caller-supplied start vector (wave-function prediction); unusable (zero, not finite) -> the random one */
        dev::d2d(st, V, d_init + R0, (size_t)N * 8);
        dev::dot(st, V, V, N, d_nrm2);
        dev::allreduce_sum(st, d_nrm2, 1);
        double n2 = 0;
        dev::d2h(st, &n2, d_nrm2, 8);
        dev::sync(st);
        have_start = std::isfinite(n2) && n2 > 1e-200;
    }
    if (!have_start) {
        dev::fill_random(st, V, N, opts.seed, R0); /* element i depends on (seed, global index) only: same start vector on any number of GPUs */
        dev::dot(st, V, V, N, d_nrm2);
        dev::allreduce_sum(st, d_nrm2, 1);
    }
    dev::scale_inv_norm(st, V, d_nrm2, V, N);

    const char* early_env = getenv("DMRGX_EARLY_TEST_MIN"); /* test hook: the size above which the in-cycle stopping test is on */
    /* ... and only where a matvec on THIS rank is long enough (>= 10 GFLOP, ~0.4 ms) to hide the host round trip of the test: on
       8 GPUs a sharded matvec of the 12x6 m = 2048 superblock takes 0.35 ms and the per-step synchronisation cost 0.3 ms
       (profiles/r2_multigpu.md) */
    /* (on several GPUs the round trip is dearer still — the NCCL operations of the next step are enqueued by the host after it —
       so the bar is twenty times higher there) */
    /* (a solve started from a predicted vector converges within a few steps of its first cycle: there the test pays from a
       tenth of that matvec size on) */
    const bool early_test = early_env ? NG >= atoll(early_env) : (NG >= 50000LL && H->alg_flops >= (dist ? 2e11 : (have_start ? 1e9 : 1e10)));
    int nc = ld, k = 0;
    double theta = 0, resid = 0;
    long long nreseed = 0;
    for (long long it = 0; it < max_it; ++it) {
        double beta_last = 0;
        bool invariant = false, reseeded = false;
        nc = ld;
        int absorbed = k; /* rows [k, absorbed) of the coefficient table are already in T */
        /* bring the coefficient rows [absorbed, upto) to the host and enter them into the projected matrix; true when an
           invariant subspace was reached after row nc - 1 (the steps queued after it worked on a null direction: their rows
           are not absorbed) */
        auto absorb_rows = [&](int upto) -> bool {
            if (upto <= absorbed) return false;
            dev::d2h(st, hh.data() + (size_t)absorbed * RW, d_tab + (size_t)absorbed * RW, (size_t)(upto - absorbed) * RW * 8);
            dev::sync(st);
            for (int j = absorbed; j < upto; ++j) {
                const double* r = hh.data() + (size_t)j * RW;
                for (int i = 0; i <= j; ++i) {
                    const double c = r[i] + r[(ld + 1) + i];
                    T[(size_t)i * ld + j] = c;
                    T[(size_t)j * ld + i] = c;
                }
                const double b = std::sqrt(std::max(0.0, r[2 * (ld + 1) + 1]));
                beta_last = b;
                if (!(b >= 1e-14)) { nc = j + 1; invariant = true; absorbed = j + 1; return true; }
            }
            absorbed = upto;
            return false;
        };
        /* classical Gram-Schmidt of w against V_0..V_{j}, twice, into V_{j+1}, with the coefficients in row j of the table: three
           fused passes over the basis with TWO reductions,
             dots  |  update + dots + ||w'||^2  |  update + normalise,
           the last norm by Pythagoras, ||w''||^2 = ||w'||^2 - |h2|^2 (the second-pass coefficients are round-off sized: no
           cancellation), so the third pass needs no reduction — on several GPUs two all-reduces per step instead of three.
           The coefficients stay on the device until the end of the cycle. */
        auto orthonormalise = [&](int j) {
            double* d_h = d_tab + (size_t)j * RW;
            double* d_h2 = d_h + (ld + 1);
            double* d_n = d_h2 + (ld + 1);   /* ||w'||^2, directly behind the pass-2 coefficients: one all-reduce covers both */
            double* d_b2 = d_n + 1;
            dev::gs_pass(st, V, N, j + 1, w, N, nullptr, d_h, nullptr);
            dev::allreduce_sum(st, d_h, j + 1);
            dev::gs_pass(st, V, N, j + 1, w, N, d_h, d_h2, d_n);
            if (dist) dev::allreduce_sum(st, d_h2, (ld + 1) + 1);
            dev::gs_final(st, V, N, j + 1, w, N, d_h2, d_n, d_b2, V + (size_t)(j + 1) * N);
        };
        for (int j0 = k;;) {
            for (int j = j0; j < nc; ++j) {
                if (dist) {
                    dev::d2d(st, xfull->as<double>() + R0, V + (size_t)j * N, (size_t)N * 8);
                    hshell_apply_sharded(H, xfull->as<double>(), w - R0);
                } else {
                    hshell_apply(H, V + (size_t)j * N, w);
                }
                stats.nmatvec++;
                orthonormalise(j);
                /* On large superblocks (a matvec costs far more than a host round trip) the stopping test is also made inside the
                   cycle, after every step from the second new one on, instead of only at the restart boundary: saves the 4 or so
                   matvecs a converged solve would otherwise still run to fill the basis. */
                if (early_test && !reseeded && j + 1 < nc && j >= k + 1) {
                    if (absorb_rows(j + 1)) break;
                    const int nj = j + 1;
                    std::vector<double> Tj((size_t)nj * nj), evj, Sj;
                    for (int a = 0; a < nj; ++a) for (int b = 0; b < nj; ++b) Tj[(size_t)a * nj + b] = T[(size_t)a * ld + b];
                    small_sym_eig(nj, Tj, evj, Sj);
                    if (std::fabs(beta_last * Sj[(size_t)(nj - 1) * nj + 0]) <= opts.tol * std::max(std::fabs(evj[0]), 1e-300)) { nc = nj; break; }
                }
            }
            if (!invariant) absorb_rows(nc);
            /* An invariant subspace smaller than the basis need not hold the wanted pair (a start vector without a ground-state
               component reaches one, e.g. an exact excited eigenvector).  As ARPACK's dgetv0 does, the cycle then goes on from a
               fresh seeded random direction, orthogonalised twice against the basis: its couplings to the exhausted block are
               round-off sized and enter T as such.  The in-cycle stopping test stays off for the rest of the cycle, so a Ritz
               pair of the exhausted block is only accepted after the new direction has had its steps. */
            if (!invariant || nc >= ld) break;
            ++nreseed;
            dev::fill_random(st, w, N, opts.seed ^ (0xD1B54A32D192ED03ULL * (unsigned long long)nreseed), R0);
            orthonormalise(nc - 1);
            invariant = false;
            reseeded = true;
            j0 = nc;
            nc = ld;
        }
        std::vector<double> Tm((size_t)nc * nc), ev, S;
        for (int i = 0; i < nc; ++i) for (int j = 0; j < nc; ++j) Tm[(size_t)i * nc + j] = T[(size_t)i * ld + j];
        small_sym_eig(nc, Tm, ev, S); /* ascending: the wanted pair is column 0 */
        theta = ev[0];
        resid = invariant ? 0.0 : std::fabs(beta_last * S[(size_t)(nc - 1) * nc + 0]);
        const bool conv = resid <= opts.tol * std::max(std::fabs(theta), 1e-300);
        const bool last = conv || (it + 1 == max_it);
        const int kk = last ? 1 : std::max(1, std::min(nc / 2, nc - 1));
        std::vector<double> Skk((size_t)nc * kk);
        for (int i = 0; i < nc; ++i) for (int a = 0; a < kk; ++a) Skk[(size_t)i * kk + a] = S[(size_t)i * nc + a];
        dev::h2d(st, d_S, Skk.data(), Skk.size() * 8);
        dev::sync(st);
        if (!last) {
            /* thick restart: V_0..V_kk-1 <- Ritz vectors, V_kk <- the residual direction */
            std::fill(T.begin(), T.end(), 0.0);
            for (int a = 0; a < kk; ++a) T[(size_t)a * ld + a] = ev[a];
            /* the residual vector sits at index nc and must survive the in-place rotation of V_0..V_nc-1 */
            dev::ritz_rotate(st, V, N, N, nc, d_S, kk);
            if (kk != nc) dev::d2d(st, V + (size_t)kk * N, V + (size_t)nc * N, (size_t)N * 8);
            k = kk;
            stats.nrestart++;
        } else {
            dev::ritz_rotate(st, V, N, N, nc, d_S, 1);
            stats.converged = conv ? 1 : 0;
            break;
        }
    }
    /* normalise the Ritz vector (it is unit up to round-off) and hand it over */
    dev::dot(st, V, V, N, d_nrm2);
    dev::allreduce_sum(st, d_nrm2, 1);
    dev::scale_inv_norm(st, V, d_nrm2, d_psi + R0, N);
    if (dist) dev::allgatherv(st, d_psi, H->row_cuts.data()); /* psi complete on every rank (the truncation reads all of it) */
    dev::sync(st);
    tr.mark("solve");
    stats.resid = resid;
    if (stats_out) *stats_out = stats;
    return theta;
}

}  // namespace dmrgx
