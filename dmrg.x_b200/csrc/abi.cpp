/*  abi.cpp — extern "C" surface declared in include/dmrgx.h.  Thin: argument marshalling, status codes,
 *  no exception crosses the boundary. */
#include <cstring>
#include <string>

#include "../../include/dmrgx.h"
#include <cmath>

#include "common.h"
#include "plan.h"

using namespace dmrgx;

namespace {
thread_local std::string g_msg;
template <class F>
int guard(F&& f) {
    try { f(); return 0; }
    catch (const Err& e) { g_msg = e.what(); return e.code ? e.code : 1; }
    catch (const std::exception& e) { g_msg = e.what(); return 1; }
    catch (...) { g_msg = "unknown error"; return 1; }
}
/* Every handle leads to its context; the context's device is made current on the way in, so that a process may hold
   contexts on several devices (allocations and launches of a context must never land on another context's GPU). */
inline Ctx* cur(Ctx* c) { if (c && c->st) dev::make_current(c->st); return c; }
inline Ctx* C(dmrgx_ctx c) { return cur((Ctx*)c); }
inline Block* B(dmrgx_block b) { if (b) cur(((Block*)b)->ctx); return (Block*)b; }
inline Kron* K(dmrgx_kron k) { if (k) cur(((Kron*)k)->ctx); return (Kron*)k; }
inline HShell* H(dmrgx_hshell h) { if (h) cur(((HShell*)h)->ctx); return (HShell*)h; }
inline XForm* X(dmrgx_xform x) { if (x) cur(((XForm*)x)->ctx); return (XForm*)x; }
std::vector<Term> terms_of(dmrgx_int n, const double* a, const int* iop, const dmrgx_int* isite, const int* jop, const dmrgx_int* jsite) {
    std::vector<Term> t;
    for (dmrgx_int i = 0; i < n; ++i) t.push_back({a[i], iop[i], isite[i], jop[i], jsite[i]});
    return t;
}
}  // namespace

extern "C" {

const char* dmrgx_last_error(void) { return g_msg.c_str(); }
dmrgx_int dmrgx_launch_count(void) { return dev::launch_count(); }

int dmrgx_ctx_create(int device, void* stream, dmrgx_ctx* out) {
    *out = nullptr;
    dev::Stream* st = nullptr;
    int e = dev::init(device, stream, &st);
    if (e) { g_msg = dev::last_error(); return e; }
    Ctx* c = new Ctx();
    c->st = st;
    *out = (dmrgx_ctx)c;
    return 0;
}
int dmrgx_dist_unique_id(void* out128) {
    int e = dev::comm_unique_id(out128);
    if (e) g_msg = dev::last_error();
    return e;
}
int dmrgx_ctx_create_dist(int device, void* stream, int rank, int world, const void* id128, dmrgx_ctx* out) {
    if (world < 1 || rank < 0 || rank >= world) { g_msg = "dmrgx_ctx_create_dist: bad rank / world"; *out = nullptr; return ERR_ARG_OUTOFRANGE; }
    int e = dmrgx_ctx_create(device, stream, out);
    if (e) return e;
    Ctx* c = C(*out);
    e = dev::comm_init(c->st, rank, world, id128);
    if (e) { g_msg = dev::last_error(); dmrgx_ctx_destroy(*out); *out = nullptr; return e; }
    c->rank = rank; c->world = world;
    return 0;
}
int dmrgx_ctx_rank(dmrgx_ctx ctx, int* rank, int* world) { *rank = C(ctx)->rank; *world = C(ctx)->world; return 0; }
int dmrgx_ctx_destroy(dmrgx_ctx ctx) {
    if (!ctx) return 0;
    return guard([&] { Ctx* c = C(ctx); dev::destroy(c->st); c->st = nullptr; delete c; }); /* (the handle is looked up ONCE: it dies here) */
}
int dmrgx_ctx_sync(dmrgx_ctx ctx) { return guard([&] { dev::sync(C(ctx)->st); }); }
int dmrgx_ctx_set_dense_threshold(dmrgx_ctx ctx, double fill) { C(ctx)->dense_fill_threshold = fill; return 0; }

int dmrgx_block_create(dmrgx_ctx ctx, dmrgx_int nsites, dmrgx_int nsectors, const double* qn, const dmrgx_int* sz, dmrgx_block* out) {
    *out = nullptr;
    return guard([&] {
        *out = (dmrgx_block)block_from_csr_begin(C(ctx), (int)nsites, std::vector<double>(qn, qn + nsectors), std::vector<long long>(sz, sz + nsectors));
    });
}
int dmrgx_block_single_site(dmrgx_ctx ctx, int spin_twice, dmrgx_block* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_block)block_single_site(C(ctx), spin_twice); });
}
int dmrgx_block_set_operator(dmrgx_block blk, int op, dmrgx_int isite, const dmrgx_int* rowptr, const dmrgx_int* colidx, const double* values) {
    return guard([&] { block_set_operator(B(blk), op, (int)isite, rowptr, colidx, values); });
}
int dmrgx_block_get_operator(dmrgx_block blk, int op, dmrgx_int isite, dmrgx_int* nnz, dmrgx_int* rowptr, dmrgx_int* colidx, double* values) {
    return guard([&] {
        std::vector<long long> rp, ci;
        std::vector<double> vv;
        block_get_operator(B(blk), op, (int)isite, rp, ci, vv);
        if (nnz) *nnz = (dmrgx_int)ci.size();
        if (colidx) {
            std::copy(rp.begin(), rp.end(), rowptr);
            std::copy(ci.begin(), ci.end(), colidx);
            std::copy(vv.begin(), vv.end(), values);
        }
    });
}
int dmrgx_block_info(dmrgx_block blk, dmrgx_int* nsites, dmrgx_int* nstates, dmrgx_int* nsectors) {
    *nsites = B(blk)->nsites; *nstates = B(blk)->sec.nstates(); *nsectors = B(blk)->sec.nsec();
    return 0;
}
int dmrgx_block_sectors(dmrgx_block blk, double* qn, dmrgx_int* sz) {
    const Sectors& s = B(blk)->sec;
    for (int i = 0; i < s.nsec(); ++i) { qn[i] = s.qn[i]; sz[i] = s.size[i]; }
    return 0;
}
int dmrgx_block_check(dmrgx_block blk) { return guard([&] { block_check(B(blk)); }); }
int dmrgx_block_destroy(dmrgx_block blk) { return guard([&] { delete B(blk); }); }
int dmrgx_block_enlarge(dmrgx_block left, dmrgx_block site, dmrgx_int nterms, const double* a, const int* iop, const dmrgx_int* isite,
                        const int* jop, const dmrgx_int* jsite, dmrgx_block* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_block)block_enlarge(B(left), B(site), terms_of(nterms, a, iop, isite, jop, jsite)); });
}

int dmrgx_kron_create(dmrgx_block left, dmrgx_block right, dmrgx_int nqn, const double* qn, dmrgx_kron* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_kron)kron_create(B(left), B(right), std::vector<double>(qn, qn + nqn)); });
}
int dmrgx_kron_destroy(dmrgx_kron k) { return guard([&] { delete K(k); }); }
dmrgx_int dmrgx_kron_size(dmrgx_kron k) { return (dmrgx_int)K(k)->pairs.size(); }
dmrgx_int dmrgx_kron_num_states(dmrgx_kron k) { return K(k)->nstates(); }
int dmrgx_kron_data(dmrgx_kron k, double* qn, dmrgx_int* li, dmrgx_int* ri, dmrgx_int* sizes, dmrgx_int* offsets) {
    const Kron* kk = K(k);
    for (size_t p = 0; p < kk->pairs.size(); ++p) { qn[p] = kk->pairs[p].qn; li[p] = kk->pairs[p].il; ri[p] = kk->pairs[p].ir; sizes[p] = kk->pairs[p].size; }
    for (size_t p = 0; p < kk->off.size(); ++p) offsets[p] = kk->off[p];
    return 0;
}
dmrgx_int dmrgx_kron_map(dmrgx_kron k, dmrgx_int l, dmrgx_int r) { return K(k)->find((int)l, (int)r); }
dmrgx_int dmrgx_kron_offsets_lr(dmrgx_kron k, dmrgx_int l, dmrgx_int r) { int p = K(k)->find((int)l, (int)r); return p < 0 ? -1 : K(k)->off[p]; }

int dmrgx_hshell_create(dmrgx_kron k, dmrgx_int nterms, const double* a, const int* iop, const dmrgx_int* isite, const int* jop,
                        const dmrgx_int* jsite, dmrgx_hshell* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_hshell)hshell_create(K(k), terms_of(nterms, a, iop, isite, jop, jsite)); });
}
int dmrgx_hshell_create_single(dmrgx_kron k, int opl, dmrgx_int il, int opr, dmrgx_int ir, dmrgx_hshell* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_hshell)hshell_create_single(K(k), opl, (int)il, opr, (int)ir); });
}
int dmrgx_hshell_create_product(dmrgx_kron k, dmrgx_int nl, const int* lop, const dmrgx_int* lsite, dmrgx_int nr, const int* rop,
                                const dmrgx_int* rsite, dmrgx_hshell* out) {
    *out = nullptr;
    return guard([&] {
        std::vector<std::pair<int, int>> l, r;
        for (dmrgx_int i = 0; i < nl; ++i) l.push_back({lop[i], (int)lsite[i]});
        for (dmrgx_int i = 0; i < nr; ++i) r.push_back({rop[i], (int)rsite[i]});
        *out = (dmrgx_hshell)hshell_create_product(K(k), l, r);
    });
}
int dmrgx_hshell_apply(dmrgx_hshell h, const double* d_x, double* d_y) { return guard([&] { hshell_apply(H(h), d_x, d_y); }); }
int dmrgx_hshell_apply_sharded(dmrgx_hshell h, double* d_x, double* d_y) { return guard([&] { hshell_apply_sharded(H(h), d_x, d_y); }); }
int dmrgx_hshell_halo_bytes(dmrgx_hshell h, double* halo, double* allgather) {
    HShell* s = H(h);
    if (halo) *halo = 8.0 * (double)s->halo_recv_elems;
    if (allgather) *allgather = 8.0 * (double)(s->n - (s->row_end - s->row_begin)) * (s->ctx->world > 1 ? 1.0 : 0.0);
    return 0;
}
int dmrgx_hshell_row_range(dmrgx_hshell h, dmrgx_int* begin, dmrgx_int* end, dmrgx_int* cuts) {
    HShell* s = H(h);
    if (begin) *begin = s->row_begin;
    if (end) *end = s->row_end;
    if (cuts) for (size_t i = 0; i < s->row_cuts.size(); ++i) cuts[i] = s->row_cuts[i];
    return 0;
}
int dmrgx_hshell_apply_stage(dmrgx_hshell h, int stage, const double* d_x, double* d_y) {
    return guard([&] {
        HShell* s = H(h);
        if (s->sparse) { if (stage == 2) hshell_apply(s, d_x, d_y); else if (stage != 1) throw Err(ERR_ARG_WRONG, "stage must be 1 or 2"); return; }
        if (stage == 1) s->stage1.run(s->ctx, d_x, nullptr);
        else if (stage == 2) s->stage2.run(s->ctx, d_x, d_y);
        else throw Err(ERR_ARG_WRONG, "stage must be 1 or 2");
    });
}
int dmrgx_hshell_stage_flops(dmrgx_hshell h, double* flops1, double* flops2) {
    *flops1 = H(h)->stage1.flops; *flops2 = H(h)->stage2.flops;
    return 0;
}
/* plan introspection (profiling aid): per work item of a stage {tm, tn, number of segments, sum of K over GEMM segments};
   returns the number of items (fills at most cap) */
dmrgx_int dmrgx_hshell_plan_items(dmrgx_hshell h, int stage, dmrgx_int cap, dmrgx_int* out4) {
    const Plan& p = stage == 1 ? H(h)->stage1 : H(h)->stage2;
    dmrgx_int n = 0;
    for (const dev::WorkItem& it : p.items) {
        if (n < cap) {
            long long ks = 0;
            for (int sgi = it.seg_begin; sgi < it.seg_end; ++sgi) if (p.segs[sgi].type == dev::SEG_GEMM) ks += p.segs[sgi].K;
            out4[4 * n] = it.tm; out4[4 * n + 1] = it.tn; out4[4 * n + 2] = it.seg_end - it.seg_begin; out4[4 * n + 3] = ks;
        }
        ++n;
    }
    return n;
}
/* plan introspection: how often each segment type (dev::SegType 0..5) is executed by the items of a stage */
int dmrgx_hshell_plan_segtypes(dmrgx_hshell h, int stage, dmrgx_int* out6) {
    const Plan& p = stage == 1 ? H(h)->stage1 : H(h)->stage2;
    for (int i = 0; i < 6; ++i) out6[i] = 0;
    for (const dev::WorkItem& it : p.items)
        for (int sgi = it.seg_begin; sgi < it.seg_end; ++sgi) out6[p.segs[sgi].type]++;
    return 0;
}
int dmrgx_hshell_stage_exec_flops(dmrgx_hshell h, double* flops1, double* flops2) {
    *flops1 = H(h)->stage1.exec_flops; *flops2 = H(h)->stage2.exec_flops;
    return 0;
}
int dmrgx_hshell_apply_host(dmrgx_hshell h, const double* x, double* y) {
    return guard([&] {
        HShell* s = H(h);
        Ctx* ctx = s->ctx;
        const size_t bytes = (size_t)s->n * 8;
        if (!s->xbuf) {
            s->xbuf = std::make_shared<DevBuf>(ctx, bytes);
            s->ybuf = std::make_shared<DevBuf>(ctx, bytes);
        }
        /* x / y are this rank's LOCAL rows (what VecGetArray gives on the reference's MPI vectors); the whole vector on one GPU */
        const size_t lbytes = (size_t)(s->row_end - s->row_begin) * 8;
        dev::h2d(ctx->st, s->xbuf->as<double>() + s->row_begin, x, lbytes);
        hshell_apply_sharded(s, s->xbuf->as<double>(), s->ybuf->as<double>());
        dev::d2h(ctx->st, y, s->ybuf->as<double>() + s->row_begin, lbytes);
        dev::sync(ctx->st);
    });
}
int dmrgx_hshell_destroy(dmrgx_hshell h) { return guard([&] { if (h) { dev::sync(H(h)->ctx->st); delete H(h); } }); }
/* device memory one apply streams through: the V workspace, the pre-summed right factors and psi in / out (the original
   operator panels come on top); what decides whether the apply can live in L2 */
int dmrgx_hshell_workspace_bytes(dmrgx_hshell h, double* bytes) {
    HShell* s = H(h);
    double b = 16.0 * (double)s->n + (s->work ? (double)s->work->bytes : 0.0);
    for (const BufRef& k : s->keep) b += (double)k->bytes;
    *bytes = b;
    return 0;
}
int dmrgx_hshell_stats_global(dmrgx_hshell h, double* alg_bytes, double* alg_flops) {
    *alg_bytes = (double)H(h)->alg_bytes_global; *alg_flops = H(h)->alg_flops_global;
    return 0;
}
int dmrgx_hshell_stats(dmrgx_hshell h, dmrgx_int* nstates, dmrgx_int* nterms, double* alg_bytes, double* alg_flops, dmrgx_int* nt1, dmrgx_int* nt2) {
    HShell* s = H(h);
    if (nstates) *nstates = s->n;
    if (nterms) *nterms = s->nterms;
    if (alg_bytes) *alg_bytes = (double)s->alg_bytes;
    if (alg_flops) *alg_flops = s->alg_flops;
    if (nt1) *nt1 = (dmrgx_int)s->stage1.items.size();
    if (nt2) *nt2 = s->sparse ? (dmrgx_int)s->sparse->tiles.size() : (dmrgx_int)s->stage2.items.size();
    return 0;
}

int dmrgx_eigs_smallest(dmrgx_hshell h, const dmrgx_eigs_opts* opts, double* e0, double* d_psi, dmrgx_eigs_stats* stats) {
    return guard([&] {
        EigsOpts o;
        if (opts) { o.tol = opts->tol; o.ncv = (int)opts->ncv; o.max_it = (int)opts->max_it; o.seed = opts->seed; }
        if (o.tol <= 0) o.tol = 1e-8;
        if (o.ncv <= 0) o.ncv = 16;
        EigsStats s;
        *e0 = eigs_smallest(H(h), o, d_psi, &s);
        if (stats) { stats->nmatvec = s.nmatvec; stats->nrestart = s.nrestart; stats->converged = s.converged; stats->resid = s.resid; }
    });
}

int dmrgx_eigs_smallest_from(dmrgx_hshell h, const dmrgx_eigs_opts* opts, const double* d_initial, double* e0, double* d_psi, dmrgx_eigs_stats* stats) {
    return guard([&] {
        EigsOpts o;
        if (opts) { o.tol = opts->tol; o.ncv = (int)opts->ncv; o.max_it = (int)opts->max_it; o.seed = opts->seed; }
        if (o.tol <= 0) o.tol = 1e-8;
        if (o.ncv <= 0) o.ncv = 16;
        EigsStats s;
        *e0 = eigs_smallest(H(h), o, d_psi, &s, d_initial);
        if (stats) { stats->nmatvec = s.nmatvec; stats->nrestart = s.nrestart; stats->converged = s.converged; stats->resid = s.resid; }
    });
}

int dmrgx_wave_create(dmrgx_kron k, const double* d_psi, dmrgx_xform grown_side, int grow_left, dmrgx_wave* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_wave)wave_create(K(k), d_psi, X(grown_side), grow_left != 0); });
}
int dmrgx_wave_apply(dmrgx_wave w, dmrgx_xform shrinking_side, dmrgx_block site, dmrgx_kron k_new, double* d_psi_new, int* ok) {
    *ok = 0;
    return guard([&] { *ok = wave_apply((const Wave*)w, X(shrinking_side), B(site), K(k_new), d_psi_new) ? 1 : 0; });
}
int dmrgx_wave_destroy(dmrgx_wave w) { return guard([&] { delete (Wave*)w; }); }

int dmrgx_truncate(dmrgx_kron k, const double* d_psi, dmrgx_int mstates, dmrgx_xform* left, dmrgx_xform* right) {
    *left = nullptr; *right = nullptr;
    return guard([&] {
        XForm *l, *r;
        truncate(K(k), d_psi, mstates, &l, &r);
        *left = (dmrgx_xform)l; *right = (dmrgx_xform)r;
    });
}
int dmrgx_xform_info(dmrgx_xform x, dmrgx_int* m, dmrgx_int* nstates, dmrgx_int* nsectors, double* trunc_err, dmrgx_int* nspec) {
    const XForm* f = X(x);
    if (m) *m = f->newsec.nstates();
    if (nstates) *nstates = f->nstates_old;
    if (nsectors) *nsectors = f->newsec.nsec();
    if (trunc_err) *trunc_err = f->trunc_err;
    if (nspec) *nspec = (dmrgx_int)f->spec_eig.size();
    return 0;
}
int dmrgx_xform_sectors(dmrgx_xform x, double* qn, dmrgx_int* sz) {
    const Sectors& s = X(x)->newsec;
    for (int i = 0; i < s.nsec(); ++i) { qn[i] = s.qn[i]; sz[i] = s.size[i]; }
    return 0;
}
int dmrgx_xform_spectrum(dmrgx_xform x, double* eigval, dmrgx_int* blk) {
    const XForm* f = X(x);
    for (size_t i = 0; i < f->spec_eig.size(); ++i) { eigval[i] = f->spec_eig[i]; blk[i] = f->spec_blk[i]; }
    return 0;
}
int dmrgx_xform_rotmat(dmrgx_xform x, double* out) {
    return guard([&] {
        const XForm* f = X(x);
        const long long m = f->newsec.nstates(), n = f->nstates_old;
        std::memset(out, 0, sizeof(double) * m * n);
        for (int k = 0; k < f->newsec.nsec(); ++k) {
            const int mk = f->newsec.size[k], nk = f->old_size[k];
            std::vector<double> u((size_t)mk * nk);
            dev::d2h(f->ctx->st, u.data(), f->U[k]->p, u.size() * 8);
            dev::sync(f->ctx->st);
            for (int i = 0; i < mk; ++i)
                std::memcpy(out + (size_t)(f->newsec.off[k] + i) * n + f->old_off[k], u.data() + (size_t)i * nk, sizeof(double) * nk);
        }
    });
}
int dmrgx_xform_destroy(dmrgx_xform x) { return guard([&] { delete X(x); }); }

int dmrgx_rotate(dmrgx_block enlarged, dmrgx_xform x, dmrgx_block* out) {
    *out = nullptr;
    return guard([&] { *out = (dmrgx_block)rotate(B(enlarged), X(x)); });
}

int dmrgx_expect(dmrgx_hshell h1, const double* d_psi, double* value) {
    return guard([&] {
        HShell* s = H(h1);
        Ctx* ctx = s->ctx;
        BufRef y = std::make_shared<DevBuf>(ctx, (size_t)s->n * 8 + 8);
        hshell_apply(s, d_psi, y->as<double>()); /* psi is complete on every rank; each computes its own rows */
        double* d_out = y->as<double>() + s->n;
        dev::dot(ctx->st, d_psi + s->row_begin, y->as<double>() + s->row_begin, s->row_end - s->row_begin, d_out);
        dev::allreduce_sum(ctx->st, d_out, 1);
        dev::d2h(ctx->st, value, d_out, 8);
        dev::sync(ctx->st);
    });
}

int dmrgx_corr_matrix(dmrgx_kron k, const double* d_psi, double* szsz, double* spsm, double* smsp, double* sz, double* flops) {
    return guard([&] { corr_matrix(K(k), d_psi, szsz, spsm, smsp, sz, flops); });
}

int dmrgx_dimer_matrix(dmrgx_kron k, const double* d_psi, dmrgx_int nbonds, const dmrgx_int* site_i, const dmrgx_int* site_j, double* dd,
                       double* d, double* flops) {
    return guard([&] { dimer_matrix(K(k), d_psi, nbonds, site_i, site_j, dd, d, flops); });
}

/* microbenchmark of the chain engine on one plain product C[M,N] = A·B (selectable operand layouts), for profiling */
int dmrgx_selftest_gemm(dmrgx_ctx cx, dmrgx_int M, dmrgx_int N, dmrgx_int K, int a_k_contig, int b_k_contig, int nseg, int reps, double* ms,
                        double* max_err) {
    return guard([&] {
        Ctx* ctx = C(cx);
        BufRef A = std::make_shared<DevBuf>(ctx, (size_t)M * K * nseg * 8), B = std::make_shared<DevBuf>(ctx, (size_t)N * K * nseg * 8),
               Cc = std::make_shared<DevBuf>(ctx, (size_t)M * N * 8);
        dev::fill_random(ctx->st, A->as<double>(), M * K * nseg, 1);
        dev::fill_random(ctx->st, B->as<double>(), N * K * nseg, 2);
        Plan plan;
        std::vector<Contribution> cs;
        for (int sgi = 0; sgi < nseg; ++sgi) {
            Contribution c;
            c.r0 = 0; c.c0 = 0; c.nr = (int)M; c.nc = (int)N;
            c.seg = make_seg(dev::SEG_GEMM);
            c.seg.A = A->as<double>() + (size_t)sgi * M * K; c.seg.B = B->as<double>() + (size_t)sgi * N * K; c.seg.K = (int)K;
            if (a_k_contig) { c.seg.lda_m = K; c.seg.lda_k = 1; } else { c.seg.lda_m = 1; c.seg.lda_k = M; }
            if (b_k_contig) { c.seg.ldb_n = K; c.seg.ldb_k = 1; } else { c.seg.ldb_n = 1; c.seg.ldb_k = N; }
            cs.push_back(c);
        }
        emit_cells(plan, Cc->as<double>(), false, N, (int)M, (int)N, cs, true);
        plan.upload(ctx);
        plan.run(ctx);
        dev::sync(ctx->st);
        const double t0 = Trace::now();
        for (int r = 0; r < reps; ++r) plan.run(ctx);
        dev::sync(ctx->st);
        *ms = (Trace::now() - t0) * 1e3 / std::max(1, reps);
        /* every element (or, for large products, every 7th row x every 5th column plus the last rows / columns of the ragged
           edge) against host dot products of the same operands */
        std::vector<double> ha((size_t)M * K * nseg), hb((size_t)N * K * nseg), hc((size_t)M * N);
        dev::d2h(ctx->st, ha.data(), A->p, ha.size() * 8); dev::d2h(ctx->st, hb.data(), B->p, hb.size() * 8);
        dev::d2h(ctx->st, hc.data(), Cc->p, hc.size() * 8);
        dev::sync(ctx->st);
        const bool full = (double)M * (double)N * (double)K * nseg <= 5e8;
        double worst = 0;
        for (long long i = 0; i < M; ++i) {
            if (!full && i % 7 != 0 && i < M - 20) continue;
            for (long long j = 0; j < N; ++j) {
                if (!full && j % 5 != 0 && j < N - 20) continue;
                double ref = 0;
                for (int sgi = 0; sgi < nseg; ++sgi) {
                    const double* pa = ha.data() + (size_t)sgi * M * K;
                    const double* pb = hb.data() + (size_t)sgi * N * K;
                    for (long long k = 0; k < K; ++k)
                        ref += (a_k_contig ? pa[i * K + k] : pa[k * M + i]) * (b_k_contig ? pb[j * K + k] : pb[k * N + j]);
                }
                worst = std::max(worst, std::fabs(ref - hc[(size_t)i * N + j]));
            }
        }
        *max_err = worst;
    });
}

int dmrgx_selftest_eig(dmrgx_ctx cx, dmrgx_int nblocks, const dmrgx_int* n, double* a, double* w, double* ms) {
    return guard([&] {
        Ctx* ctx = C(cx);
        long long tot = 0, wtot = 0;
        for (dmrgx_int b = 0; b < nblocks; ++b) { tot += n[b] * n[b]; wtot += n[b]; }
        BufRef A = std::make_shared<DevBuf>(ctx, (size_t)std::max<long long>(1, tot) * 8), W = std::make_shared<DevBuf>(ctx, (size_t)std::max<long long>(1, wtot) * 8);
        dev::h2d(ctx->st, A->p, a, (size_t)tot * 8);
        std::vector<int> nn; std::vector<double*> pa, pw;
        long long oa = 0, ow = 0;
        for (dmrgx_int b = 0; b < nblocks; ++b) { nn.push_back((int)n[b]); pa.push_back(A->as<double>() + oa); pw.push_back(W->as<double>() + ow); oa += n[b] * n[b]; ow += n[b]; }
        dev::sync(ctx->st);
        const double t0 = Trace::now();
        const int e = dev::syevd_batch(ctx->st, (int)nblocks, nn.data(), pa.data(), pw.data());
        dev::sync(ctx->st);
        if (ms) *ms = (Trace::now() - t0) * 1e3;
        if (e) throw Err(ERR_GENERIC, std::string("eigensolver failed: ") + dev::last_error());
        dev::d2h(ctx->st, a, A->p, (size_t)tot * 8);
        dev::d2h(ctx->st, w, W->p, (size_t)wtot * 8);
        dev::sync(ctx->st);
    });
}

dmrgx_int dmrgx_ham_terms(dmrgx_int Lx, dmrgx_int Ly, double J1, double Jz1, double J2, double Jz2, int bcx, int bcy, dmrgx_int nsites,
                          dmrgx_int maxterms, double* a, int* iop, dmrgx_int* isite, int* jop, dmrgx_int* jsite) {
    std::vector<Term> t = ham_terms(Lx, Ly, J1, Jz1, J2, Jz2, bcx, bcy, nsites);
    for (dmrgx_int i = 0; i < (dmrgx_int)t.size() && i < maxterms; ++i) {
        a[i] = t[i].a; iop[i] = t[i].Iop; isite[i] = t[i].Isite; jop[i] = t[i].Jop; jsite[i] = t[i].Jsite;
    }
    return (dmrgx_int)t.size();
}

int dmrgx_vec_alloc(dmrgx_ctx ctx, dmrgx_int n, double** d_out) { return guard([&] { *d_out = (double*)dev::malloc_bytes(C(ctx)->st, (size_t)n * 8); }); }
int dmrgx_vec_free(dmrgx_ctx ctx, double* d) { return guard([&] { dev::free_bytes(C(ctx)->st, d); }); }
int dmrgx_vec_set(dmrgx_ctx ctx, double* d_dst, const double* h_src, dmrgx_int n) {
    return guard([&] { dev::h2d(C(ctx)->st, d_dst, h_src, (size_t)n * 8); dev::sync(C(ctx)->st); });
}
int dmrgx_vec_get(dmrgx_ctx ctx, double* h_dst, const double* d_src, dmrgx_int n) {
    return guard([&] { dev::d2h(C(ctx)->st, h_dst, d_src, (size_t)n * 8); dev::sync(C(ctx)->st); });
}

}  // extern "C"
