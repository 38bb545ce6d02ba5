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
 */
#include <algorithm>
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

}  // namespace dmrgx
