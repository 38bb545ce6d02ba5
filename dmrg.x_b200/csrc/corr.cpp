/*  corr.cpp — EXTENSION: every two-point spin correlator, and every bond–bond (dimer) correlator over a bond list, of the
 *  superblock in one batched pass each.
 *
 *  For single-site operators O_a, O_b:  <psi| O_a O_b |psi> = < O_a† psi , O_b psi >,  so the whole matrix is a Gram matrix of
 *  single-operator panels  Pi_t[s] = (O_t at superblock site s) psi  — one group per operator type t in {Sz, S-, S+}:
 *      SzSz[i][j] = <Sz_i psi, Sz_j psi>             (psi itself is the last column of the Sz group: Sz_i = <psi, Sz_i psi>)
 *      SpSm[i][j] = <psi| S+_i S-_j |psi> = <S-_i psi, S-_j psi>     panels in the sector qn - 1
 *      SmSp[i][j] = <psi| S-_i S+_j |psi> = <S+_i psi, S+_j psi>     panels in the sector qn + 1
 *  A left-block panel is A·X_q per sector pair (stage 1 of H·psi), a right-block one X_q·Bᵀ (stage 2), laid out as the Kron of
 *  the shifted sector.  All panels of a group are ONE chain-kernel plan (one launch), followed by one dev::gram; each group's
 *  buffer is freed before the next one is built.  Same-block entries are products of the block's own operators in list
 *  order, exactly what hshell_create_product computes; cross-block entries are <A_i ⊗ B_j>.
 *
 *  The dimer matrix is the Gram matrix of the bond panels  D̃_a psi = Sz_i (Sz_j psi) + ½ S+_i (S-_j psi) + ½ S-_i (S+_j psi)
 *  (bond a = (i, j) in the caller's order), built in two chain-kernel plans: the single-operator panels of every second site j
 *  in all three sectors, then every bond panel as the sum of its three terms in psi's sector.
 *
 *  The spectral recurrence (continued-fraction method, K. Hallberg, PRB 52, R9827 (1995)) starts from  phi_v = Σ_s coef[v][s] O_s psi
 *  in the sector qn + op: the n single-operator panels are one chain-kernel plan, the start vectors of a batch are one GEMM
 *  plan  Phi = C·P  over them, and every vector then runs a plain three-term Lanczos recurrence of the target shell, the whole
 *  batch advanced by dev::lanczos_batch with no host synchronisation until the batch is finished.  With overlaps, every step
 *  also takes the rectangular Gram block <O_s psi, v_t> of the n panels against the batch's freshly normalised Lanczos vectors
 *  (dev::gram_rect), from which any matrix element <O_s psi| f(H) |phi_v> follows on the host.
 */
#include <algorithm>
#include <cmath>
#include <memory>
#include <set>
#include <string>

#include "common.h"
#include "plan.h"

namespace dmrgx {

/* One term  coef · O · src  of a panel: O acts on one block (left: A ⊗ 1, right: 1 ⊗ B) and src is laid out as `src_kron`, a
   Kron of the same two blocks in any sector. */
struct PanelTerm {
    bool left;
    const Operator* O;
    const Kron* src_kron;
    const double* src;
    double coef;
};

/* Appends the contributions of one term to output pair p of `out_kron` (none when the term does not reach that pair). */
static void term_contributions(std::vector<Contribution>& cs, const Kron* out_kron, size_t p, const PanelTerm& t) {
    const Kron* sk = t.src_kron;
    const Sectors &SL = out_kron->L->sec, &SR = out_kron->R->sec;
    const int il = out_kron->pairs[p].il, ir = out_kron->pairs[p].ir;
    const int nL = SL.size[il], nR = SR.size[ir];
    if (t.left) {   /* (A ⊗ 1) X:  Y(il, ir) = A[il, jl] · X(jl, ir) */
        const int jl = il + t.O->shift;
        const int q = (jl >= 0 && jl < SL.nsec()) ? sk->find(jl, ir) : -1;
        if (q < 0) return;
        for (const Tile& a : t.O->tiles[il]) {
            const double* X = t.src + sk->off[q] + (long long)(a.c0 - SL.off[jl]) * nR;
            Contribution c;
            c.r0 = a.r0 - SL.off[il]; c.nr = a.nr; c.c0 = 0; c.nc = nR;
            if (a.fmt == T_DENSE) {
                c.seg = make_seg(dev::SEG_GEMM);
                c.seg.A = a.d; c.seg.lda_m = a.sr; c.seg.lda_k = a.sc; c.seg.K = a.nc;
                c.seg.B = X; c.seg.ldb_k = nR; c.seg.ldb_n = 1; c.seg.coef = t.coef;
            } else if (a.fmt == T_EYE) {
                c.seg = make_seg(dev::SEG_AXPY);
                c.seg.A = X; c.seg.lda_m = nR; c.seg.lda_k = 1; c.seg.coef = a.scale * t.coef;
            } else {
                c.seg = make_seg(dev::SEG_CSRA);
                c.seg.rowptr = a.rowptr; c.seg.colidx = a.col; c.seg.B = a.val;
                c.seg.A = X; c.seg.ldb_k = nR; c.seg.ldb_n = 1; c.seg.coef = t.coef;
            }
            cs.push_back(c);
        }
    } else {        /* (1 ⊗ B) X:  Y(il, ir) = X(il, jr) · B[ir, jr]ᵀ */
        const int jr = ir + t.O->shift;
        const int q = (jr >= 0 && jr < SR.nsec()) ? sk->find(il, jr) : -1;
        if (q < 0) return;
        const int nRq = SR.size[jr];
        for (const Tile& b : t.O->tiles[ir]) {
            const double* X = t.src + sk->off[q] + (b.c0 - SR.off[jr]);
            Contribution c;
            c.r0 = 0; c.nr = nL; c.c0 = b.r0 - SR.off[ir]; c.nc = b.nr;
            if (b.fmt == T_DENSE) {
                c.seg = make_seg(dev::SEG_GEMM);
                c.seg.A = X; c.seg.lda_m = nRq; c.seg.lda_k = 1; c.seg.K = b.nc;
                c.seg.B = b.d; c.seg.ldb_n = b.sr; c.seg.ldb_k = b.sc; c.seg.coef = t.coef;
            } else if (b.fmt == T_EYE) {
                c.seg = make_seg(dev::SEG_AXPY);
                c.seg.A = X; c.seg.lda_m = nRq; c.seg.lda_k = 1; c.seg.coef = b.scale * t.coef;
            } else {
                c.seg = make_seg(dev::SEG_CSRB);
                c.seg.A = X; c.seg.lda_m = nRq; c.seg.lda_k = 1;
                c.seg.rowptr = b.rowptr; c.seg.colidx = b.col; c.seg.B = b.val; c.seg.coef = t.coef;
            }
            cs.push_back(c);
        }
    }
}

/* Panel Σ_t coef_t · O_t · src_t into the layout of `out_kron`.  All terms of one output sector pair go to ONE emit_cells call,
   so every element of the panel is written exactly once (pairs no term reaches, or sector rows no operator reaches, are
   zero-filled by the plan). */
static void plan_panel(Plan& plan, const Kron* out_kron, const std::vector<PanelTerm>& terms, double* out) {
    const Sectors &SL = out_kron->L->sec, &SR = out_kron->R->sec;
    for (size_t p = 0; p < out_kron->pairs.size(); ++p) {
        const int nL = SL.size[out_kron->pairs[p].il], nR = SR.size[out_kron->pairs[p].ir];
        if (nL == 0 || nR == 0) continue;
        std::vector<Contribution> cs;
        for (const PanelTerm& t : terms) term_contributions(cs, out_kron, p, t);
        emit_cells(plan, out + out_kron->off[p], false, nR, nL, nR, cs, true);
    }
}

/* the total Sz of a superblock that must have exactly one sector */
static double single_sector(const Kron* kron, const char* what) {
    std::set<double> qns;
    for (const KronPair& p : kron->pairs) qns.insert(p.qn);
    if (qns.size() != 1)
        throw Err(ERR_SUP, std::string(what) + " needs a superblock of exactly one total-Sz sector (this one has " + std::to_string(qns.size()) + ").");
    return *qns.begin();
}

/* superblock site s: left-block site s, or right-block site nL + nR - 1 - s (hshell_create, SetUpCorrelation) */
static const Operator* site_op(const Kron* kron, int s, int type) {
    const int nL = kron->L->nsites, n = nL + kron->R->nsites;
    return s < nL ? kron->L->op(type, s) : kron->R->op(type, n - 1 - s);
}

static void require_site_ops(const Kron* kron, int s) {
    const int nL = kron->L->nsites, n = nL + kron->R->nsites;
    if (!site_op(kron, s, OP_SZ)->present || !site_op(kron, s, OP_SP)->present)
        throw Err(ERR_ARG_WRONGSTATE, "superblock site " + std::to_string(s) + " (" + (s < nL ? "left" : "right") + " block site " +
                                          std::to_string(s < nL ? s : n - 1 - s) + "): Sz or Sp has not been set.");
}

void corr_matrix(const Kron* kron, const double* d_psi, double* szsz, double* spsm, double* smsp, double* sz, double* flops) {
    if (!d_psi) throw Err(ERR_ARG_WRONG, "psi is NULL.");
    if (!szsz || !spsm || !smsp || !sz) throw Err(ERR_ARG_WRONG, "an output matrix is NULL.");
    const double qn = single_sector(kron, "the correlation matrix");
    Ctx* ctx = kron->ctx;
    const Block *L = kron->L, *R = kron->R;
    const int nL = L->nsites, nR = R->nsites, n = nL + nR;
    for (int s = 0; s < n; ++s) require_site_ops(kron, s);
    double total = 0;
    const struct { int type; double* out; } groups[3] = {{OP_SZ, szsz}, {OP_SM, spsm}, {OP_SP, smsp}};
    for (const auto& grp : groups) {
        /* psi's own sector for Sz (the superblock itself), else the Kron of qn ± 1 */
        std::unique_ptr<Kron> shifted;
        const Kron* ok = kron;
        if (grp.type != OP_SZ) { shifted.reset(kron_create(L, R, {qn + grp.type})); ok = shifted.get(); }
        const long long D = ok->nstates();
        const int np = n + (grp.type == OP_SZ ? 1 : 0);
        std::vector<double> G((size_t)np * np, 0.0);
        if (D > 0) {
            const long long ldp = (D + 1) & ~1LL; /* every column 16-byte aligned */
            BufRef buf = std::make_shared<DevBuf>(ctx, (size_t)np * ldp * 8);
            BufRef dG = std::make_shared<DevBuf>(ctx, (size_t)np * np * 8);
            double* P = buf->as<double>();
            Plan plan;
            for (int s = 0; s < n; ++s) plan_panel(plan, ok, {{s < nL, site_op(kron, s, grp.type), kron, d_psi, 1.0}}, P + (long long)s * ldp);
            plan.upload(ctx);
            plan.run(ctx);
            if (grp.type == OP_SZ) dev::d2d(ctx->st, P + (long long)n * ldp, d_psi, (size_t)D * 8);
            dev::gram(ctx->st, P, ldp, np, D, dG->as<double>());
            dev::d2h(ctx->st, G.data(), dG->p, G.size() * 8);
            dev::sync(ctx->st); /* the plan's device lists and the panel buffer die with this scope */
            total += plan.flops + 2.0 * np * np * (double)D;
        }
        for (int i = 0; i < n; ++i)
            std::copy(G.begin() + (size_t)i * np, G.begin() + (size_t)i * np + n, grp.out + (size_t)i * n);
        if (grp.type == OP_SZ)
            for (int i = 0; i < n; ++i) sz[i] = G[(size_t)i * np + n];
    }
    if (flops) *flops = total;
}

/* The panels are built as E_a = 2·D̃_a psi: the level-1 Sz panels carry the factor 2, so every GEMM segment of the bond panels
   has a unit coefficient and takes the chain kernel's full-tile body (a coefficient other than 1 never does).  Scaling by a
   power of two is exact, so the Gram of the E_a times ¼ (and the psi column times ½) has the bits of the plain form. */
void dimer_matrix(const Kron* kron, const double* d_psi, long long nb, const long long* bond_i, const long long* bond_j, double* dd, double* d,
                  double* flops) {
    if (!d_psi) throw Err(ERR_ARG_WRONG, "psi is NULL.");
    if (!bond_i || !bond_j) throw Err(ERR_ARG_WRONG, "a bond site array is NULL.");
    if (!dd || !d) throw Err(ERR_ARG_WRONG, "an output array is NULL.");
    if (nb < 1) throw Err(ERR_ARG_OUTOFRANGE, "the dimer matrix needs at least one bond (got " + std::to_string(nb) + ").");
    const Block *L = kron->L, *R = kron->R;
    const int nL = L->nsites, n = nL + R->nsites;
    for (long long a = 0; a < nb; ++a) {
        if (bond_i[a] < 0 || bond_i[a] >= n || bond_j[a] < 0 || bond_j[a] >= n || bond_i[a] == bond_j[a])
            throw Err(ERR_ARG_OUTOFRANGE, "bond " + std::to_string(a) + " = (" + std::to_string(bond_i[a]) + ", " + std::to_string(bond_j[a]) +
                                              "): the sites must be two different superblock sites in [0, " + std::to_string(n) + ").");
    }
    const double qn = single_sector(kron, "the dimer matrix");
    /* the level-1 panels are built for the second sites only: slot[j] is j's column in each level-1 buffer */
    std::vector<char> used(n, 0);
    std::vector<int> slot(n, -1);
    int nj = 0;
    for (long long a = 0; a < nb; ++a) {
        used[bond_i[a]] = used[bond_j[a]] = 1;
        if (slot[bond_j[a]] < 0) slot[bond_j[a]] = nj++;
    }
    for (int s = 0; s < n; ++s)
        if (used[s]) require_site_ops(kron, s);
    Ctx* ctx = kron->ctx;
    const std::unique_ptr<Kron> km(kron_create(L, R, {qn - 1})), kp(kron_create(L, R, {qn + 1}));
    const long long D = kron->nstates(), Dm = km->nstates(), Dp = kp->nstates();
    const int np = (int)nb + 1;
    std::vector<double> G((size_t)np * np, 0.0);
    double total = 0;
    if (D > 0) {
        /* every column 16-byte aligned */
        const long long ld = (D + 1) & ~1LL, ldm = (Dm + 1) & ~1LL, ldq = (Dp + 1) & ~1LL;
        BufRef Q = std::make_shared<DevBuf>(ctx, (size_t)np * ld * 8), dG = std::make_shared<DevBuf>(ctx, (size_t)np * np * 8);
        {
            /* level 1: 2·Sz_j psi (sector qn), S-_j psi (qn - 1), S+_j psi (qn + 1); an empty shifted sector has no panels */
            BufRef Pz = std::make_shared<DevBuf>(ctx, (size_t)nj * ld * 8);
            BufRef Pm = Dm > 0 ? std::make_shared<DevBuf>(ctx, (size_t)nj * ldm * 8) : nullptr;
            BufRef Pp = Dp > 0 ? std::make_shared<DevBuf>(ctx, (size_t)nj * ldq * 8) : nullptr;
            auto col = [&](const BufRef& b, long long ldb, int s) { return b->as<double>() + (long long)slot[s] * ldb; };
            Plan level1, level2;
            for (int s = 0; s < n; ++s) {
                if (slot[s] < 0) continue;
                plan_panel(level1, kron, {{s < nL, site_op(kron, s, OP_SZ), kron, d_psi, 2.0}}, col(Pz, ld, s));
                if (Pm) plan_panel(level1, km.get(), {{s < nL, site_op(kron, s, OP_SM), kron, d_psi, 1.0}}, col(Pm, ldm, s));
                if (Pp) plan_panel(level1, kp.get(), {{s < nL, site_op(kron, s, OP_SP), kron, d_psi, 1.0}}, col(Pp, ldq, s));
            }
            /* level 2: E_a = Sz_i (2 Sz_j psi) + S+_i (S-_j psi) + S-_i (S+_j psi), one output panel per bond in sector qn */
            for (long long a = 0; a < nb; ++a) {
                const int i = (int)bond_i[a], j = (int)bond_j[a];
                std::vector<PanelTerm> terms = {{i < nL, site_op(kron, i, OP_SZ), kron, col(Pz, ld, j), 1.0}};
                if (Pm) terms.push_back({i < nL, site_op(kron, i, OP_SP), km.get(), col(Pm, ldm, j), 1.0});
                if (Pp) terms.push_back({i < nL, site_op(kron, i, OP_SM), kp.get(), col(Pp, ldq, j), 1.0});
                plan_panel(level2, kron, terms, Q->as<double>() + a * ld);
            }
            level1.upload(ctx);
            level2.upload(ctx);
            level1.run(ctx);
            level2.run(ctx);
            dev::d2d(ctx->st, Q->as<double>() + nb * ld, d_psi, (size_t)D * 8);
            total += level1.flops + level2.flops;
        }   /* the level-1 panels and both plans are released here: the heap is stream-ordered, the Gram runs behind them */
        dev::gram(ctx->st, Q->as<double>(), ld, np, D, dG->as<double>());
        dev::d2h(ctx->st, G.data(), dG->p, G.size() * 8);
        dev::sync(ctx->st);
        total += 2.0 * np * np * (double)D;
    }
    for (long long a = 0; a < nb; ++a) {
        for (long long b = 0; b < nb; ++b) dd[a * nb + b] = 0.25 * G[(size_t)(a * np + b)];
        d[a] = 0.5 * G[(size_t)(a * np + nb)];
    }
    if (flops) *flops = total;
}

/* Device memory for the three recurrence columns (v_prev, v, H·v) of a batch: it holds as many vectors as fit, at least one */
constexpr double SPECTRAL_BATCH_BYTES = 2.0 * (1LL << 30);
/* a start vector whose norm is at most this fraction of Σ_s |coef_s|·‖O_s psi‖ is zero up to rounding: norm2 = 0, no steps */
constexpr double SPECTRAL_ZERO_REL = 1e-12;

void spectral_lanczos(const Kron* kron, const double* d_psi, HShell* h, int op, long long nvec, const double* coef, long long nsteps,
                      double* alpha, double* beta, double* norm2, long long* nsteps_done, double* overlaps, double* flops) {
    if (!d_psi) throw Err(ERR_ARG_WRONG, "psi is NULL.");
    if (!h) throw Err(ERR_ARG_WRONG, "the target shell is NULL.");
    if (!coef) throw Err(ERR_ARG_WRONG, "the coefficient array is NULL.");
    if (!alpha || !beta || !norm2 || !nsteps_done) throw Err(ERR_ARG_WRONG, "an output array is NULL.");
    if (op != OP_SZ && op != OP_SP && op != OP_SM)
        throw Err(ERR_ARG_OUTOFRANGE, "op must be DMRGX_OP_SZ, DMRGX_OP_SP or DMRGX_OP_SM (got " + std::to_string(op) + ").");
    if (nvec < 1) throw Err(ERR_ARG_OUTOFRANGE, "the spectral recurrence needs at least one vector (got " + std::to_string(nvec) + ").");
    if (nsteps < 1) throw Err(ERR_ARG_OUTOFRANGE, "the spectral recurrence needs at least one step (got " + std::to_string(nsteps) + ").");
    const Block *L = kron->L, *R = kron->R;
    const int nL = L->nsites, n = nL + R->nsites;
    for (long long i = 0; i < nvec * n; ++i)
        if (!std::isfinite(coef[i]))
            throw Err(ERR_ARG_OUTOFRANGE, "coefficient " + std::to_string(i % n) + " of vector " + std::to_string(i / n) + " is not finite.");
    const double qn = single_sector(kron, "the spectral recurrence");
    Ctx* ctx = kron->ctx;
    if (ctx->world > 1) throw Err(ERR_SUP, "the spectral recurrence needs a single-GPU context: the sharded apply of the target shell is collective.");
    const Kron* tk = h->kron;
    std::set<double> tq;
    for (const KronPair& p : tk->pairs) tq.insert(p.qn);
    if (tk->L != L || tk->R != R || tq.size() != 1 || *tq.begin() != qn + op)
        throw Err(ERR_ARG_WRONGSTATE, "the target shell must be built on a Kron of the same two blocks whose single sector is qn + op = " +
                                          std::to_string(qn + op) + ".");
    /* the overlaps are taken against every site's panel, so each site then needs its operators */
    std::vector<char> used(n, overlaps ? 1 : 0);
    for (long long i = 0; i < nvec * n; ++i)
        if (coef[i] != 0.0) used[i % n] = 1;
    for (int s = 0; s < n; ++s)
        if (used[s]) require_site_ops(kron, s);
    std::fill(alpha, alpha + nvec * nsteps, 0.0);
    std::fill(beta, beta + nvec * nsteps, 0.0);
    std::fill(norm2, norm2 + nvec, 0.0);
    std::fill(nsteps_done, nsteps_done + nvec, 0LL);
    if (overlaps) std::fill(overlaps, overlaps + nvec * nsteps * n, 0.0);
    const long long D = tk->nstates(), ld = (D + 1) & ~1LL;
    double total = 0;
    if (D > 0) {
        dev::Stream* st = ctx->st;
        /* the n single-operator panels O_s psi in the sector qn + op, one plan; a site no vector uses is a zero column, so the
           GEMM below always runs over all n sites and a vector's bits do not depend on the others */
        BufRef Pb = std::make_shared<DevBuf>(ctx, (size_t)n * ld * 8), Cb = std::make_shared<DevBuf>(ctx, (size_t)(nvec * n) * 8);
        BufRef pnb = std::make_shared<DevBuf>(ctx, (size_t)n * 8);
        double* P = Pb->as<double>();
        dev::h2d(st, Cb->p, coef, (size_t)(nvec * n) * 8);
        Plan panels;
        for (int s = 0; s < n; ++s) {
            if (used[s]) plan_panel(panels, tk, {{s < nL, site_op(kron, s, op), kron, d_psi, 1.0}}, P + (long long)s * ld);
            else dev::memset0(st, P + (long long)s * ld, (size_t)ld * 8);
        }
        panels.upload(ctx);
        panels.run(ctx);
        total += panels.flops;
        /* ‖O_s psi‖: the scale below which a start vector is rounding noise */
        std::vector<double> pn2(n, 0.0);
        for (int s = 0; s < n; ++s)
            if (used[s]) dev::dot(st, P + (long long)s * ld, P + (long long)s * ld, D, pnb->as<double>() + s);
        dev::d2h(st, pn2.data(), pnb->p, (size_t)n * 8);
        dev::sync(st);
        for (int s = 0; s < n; ++s) pn2[s] = used[s] ? std::sqrt(pn2[s]) : 0.0;

        const int nb = (int)std::max<long long>(1, std::min<long long>(nvec, (long long)(SPECTRAL_BATCH_BYTES / (3.0 * 8.0 * (double)ld))));
        const int nblk = dev::lanczos_blocks(D);
        BufRef slots = std::make_shared<DevBuf>(ctx, (size_t)3 * nb * ld * 8);
        BufRef scal = std::make_shared<DevBuf>(ctx, (size_t)(2 * nb * nsteps + 4 * nb + (long long)nb * nblk) * 8);
        BufRef ints = std::make_shared<DevBuf>(ctx, (size_t)nb * (8 + 4 + 4));
        double* slot[3] = {slots->as<double>(), slots->as<double>() + (long long)nb * ld, slots->as<double>() + 2LL * nb * ld};
        dev::LanczosBatch lb;
        lb.nsteps = (int)nsteps; lb.n = D; lb.ld = ld;
        lb.alpha = scal->as<double>(); lb.beta = lb.alpha + (long long)nb * nsteps;
        lb.norm2 = lb.beta + (long long)nb * nsteps; lb.a = lb.norm2 + nb; lb.scale = lb.a + nb;
        double* zero2 = lb.scale + nb;
        lb.zero2 = zero2; lb.partials = zero2 + nb;
        lb.ndone = ints->as<long long>(); lb.done = (int*)(lb.ndone + nb); lb.tickets = (unsigned int*)(lb.done + nb);
        dev::memset0(st, lb.tickets, (size_t)nb * 4);
        /* overlaps of a batch on the device, [c][t][s]: column c of step t's Gram block at ov + t·n, stride nsteps·n */
        BufRef ovb = overlaps ? std::make_shared<DevBuf>(ctx, (size_t)((long long)nb * nsteps * n) * 8) : nullptr;
        std::vector<double> hz(nb);
        for (long long b0 = 0; b0 < nvec; b0 += nb) {
            const int m = (int)std::min<long long>(nb, nvec - b0);
            lb.nb = m;
            for (int c = 0; c < m; ++c) {
                double sig = 0;
                for (int s = 0; s < n; ++s) sig += std::fabs(coef[(b0 + c) * n + s]) * pn2[s];
                hz[c] = (SPECTRAL_ZERO_REL * sig) * (SPECTRAL_ZERO_REL * sig);
            }
            dev::h2d(st, zero2, hz.data(), (size_t)m * 8);
            dev::memset0(st, lb.alpha, (size_t)2 * nb * nsteps * 8);
            dev::memset0(st, lb.ndone, (size_t)nb * (8 + 4));
            /* start vectors: Phi[c] = Σ_s coef[b0 + c][s] P_s, one GEMM plan (the chain engine's plain product) into the y slot */
            int ip = 0, ic = 1, iy = 2;
            Plan comb;
            Contribution g;
            g.r0 = 0; g.c0 = 0; g.nr = m; g.nc = (int)D;
            g.seg = make_seg(dev::SEG_GEMM);
            g.seg.A = Cb->as<double>() + b0 * n; g.seg.lda_m = n; g.seg.lda_k = 1; g.seg.K = n;
            g.seg.B = P; g.seg.ldb_k = ld; g.seg.ldb_n = 1;
            emit_cells(comb, slot[iy], false, ld, m, (int)D, {g}, true);
            comb.upload(ctx);
            comb.run(ctx);
            total += comb.flops;
            auto rotate = [&] { const int p = ip; ip = ic; ic = iy; iy = p; };
            dev::lanczos_batch(st, lb, 0, -1, slot[ip], slot[ic], slot[iy]);
            rotate();
            for (long long t = 0; t < nsteps; ++t) {
                for (int c = 0; c < m; ++c) hshell_apply(h, slot[ic] + (long long)c * ld, slot[iy] + (long long)c * ld);
                dev::lanczos_batch(st, lb, 1, (int)t, slot[ip], slot[ic], slot[iy]);
                /* pass 1 has just normalised v_t in place; a done column's slot is stale, and only its own entries see it */
                if (overlaps) dev::gram_rect(st, P, ld, n, slot[ic], ld, m, D, ovb->as<double>() + t * n, 1, nsteps * n);
                if (t + 1 < nsteps) {
                    dev::lanczos_batch(st, lb, 2, (int)t, slot[ip], slot[ic], slot[iy]);
                    rotate();
                }
            }
            dev::d2h(st, alpha + b0 * nsteps, lb.alpha, (size_t)m * nsteps * 8);
            dev::d2h(st, beta + b0 * nsteps, lb.beta, (size_t)m * nsteps * 8);
            dev::d2h(st, norm2 + b0, lb.norm2, (size_t)m * 8);
            dev::d2h(st, nsteps_done + b0, lb.ndone, (size_t)m * 8);
            if (overlaps) dev::d2h(st, overlaps + b0 * nsteps * n, ovb->p, (size_t)((long long)m * nsteps * n) * 8);
            dev::sync(st); /* the combine plan and hz are reused by the next batch */
            if (overlaps)
                for (long long c = b0; c < b0 + m; ++c)
                    std::fill(overlaps + (c * nsteps + nsteps_done[c]) * n, overlaps + (c + 1) * nsteps * n, 0.0);
        }
        total += (double)nvec * (double)nsteps * h->alg_flops + (double)nvec * (10.0 * (double)nsteps + 2.0) * (double)D;
        if (overlaps) total += (double)nvec * (double)nsteps * 2.0 * (double)n * (double)D;
    }
    if (flops) *flops = total;
}

}  // namespace dmrgx
