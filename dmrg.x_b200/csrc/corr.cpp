/*  corr.cpp — EXTENSION: every two-point spin correlator of the superblock in one batched pass.
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
 */
#include <algorithm>
#include <memory>
#include <set>
#include <string>

#include "common.h"
#include "plan.h"

namespace dmrgx {

/* Panel O·psi of one superblock site into the layout of `out_kron` (the shifted sector): every element of the panel is written
   (pairs without a source, or sector rows the operator does not reach, are zero-filled by the plan). */
static void plan_panel(Plan& plan, const Kron* kron, const Kron* out_kron, bool left, const Operator* O, const double* psi, double* out) {
    const Sectors &SL = kron->L->sec, &SR = kron->R->sec;
    for (size_t p = 0; p < out_kron->pairs.size(); ++p) {
        const int il = out_kron->pairs[p].il, ir = out_kron->pairs[p].ir;
        const int nL = SL.size[il], nR = SR.size[ir];
        if (nL == 0 || nR == 0) continue;
        std::vector<Contribution> cs;
        if (left) {   /* (A ⊗ 1) psi:  Y(il, ir) = A[il, jl] · X(jl, ir) */
            const int jl = il + O->shift;
            const int q = (jl >= 0 && jl < SL.nsec()) ? kron->find(jl, ir) : -1;
            if (q >= 0)
                for (const Tile& a : O->tiles[il]) {
                    const double* X = psi + kron->off[q] + (long long)(a.c0 - SL.off[jl]) * nR;
                    Contribution c;
                    c.r0 = a.r0 - SL.off[il]; c.nr = a.nr; c.c0 = 0; c.nc = nR;
                    if (a.fmt == T_DENSE) {
                        c.seg = make_seg(dev::SEG_GEMM);
                        c.seg.A = a.d; c.seg.lda_m = a.sr; c.seg.lda_k = a.sc; c.seg.K = a.nc;
                        c.seg.B = X; c.seg.ldb_k = nR; c.seg.ldb_n = 1;
                    } else if (a.fmt == T_EYE) {
                        c.seg = make_seg(dev::SEG_AXPY);
                        c.seg.A = X; c.seg.lda_m = nR; c.seg.lda_k = 1; c.seg.coef = a.scale;
                    } else {
                        c.seg = make_seg(dev::SEG_CSRA);
                        c.seg.rowptr = a.rowptr; c.seg.colidx = a.col; c.seg.B = a.val;
                        c.seg.A = X; c.seg.ldb_k = nR; c.seg.ldb_n = 1;
                    }
                    cs.push_back(c);
                }
        } else {      /* (1 ⊗ B) psi:  Y(il, ir) = X(il, jr) · B[ir, jr]ᵀ */
            const int jr = ir + O->shift;
            const int q = (jr >= 0 && jr < SR.nsec()) ? kron->find(il, jr) : -1;
            if (q >= 0) {
                const int nRq = SR.size[jr];
                for (const Tile& b : O->tiles[ir]) {
                    const double* X = psi + kron->off[q] + (b.c0 - SR.off[jr]);
                    Contribution c;
                    c.r0 = 0; c.nr = nL; c.c0 = b.r0 - SR.off[ir]; c.nc = b.nr;
                    if (b.fmt == T_DENSE) {
                        c.seg = make_seg(dev::SEG_GEMM);
                        c.seg.A = X; c.seg.lda_m = nRq; c.seg.lda_k = 1; c.seg.K = b.nc;
                        c.seg.B = b.d; c.seg.ldb_n = b.sr; c.seg.ldb_k = b.sc;
                    } else if (b.fmt == T_EYE) {
                        c.seg = make_seg(dev::SEG_AXPY);
                        c.seg.A = X; c.seg.lda_m = nRq; c.seg.lda_k = 1; c.seg.coef = b.scale;
                    } else {
                        c.seg = make_seg(dev::SEG_CSRB);
                        c.seg.A = X; c.seg.lda_m = nRq; c.seg.lda_k = 1;
                        c.seg.rowptr = b.rowptr; c.seg.colidx = b.col; c.seg.B = b.val;
                    }
                    cs.push_back(c);
                }
            }
        }
        emit_cells(plan, out + out_kron->off[p], false, nR, nL, nR, cs, true);
    }
}

void corr_matrix(const Kron* kron, const double* d_psi, double* szsz, double* spsm, double* smsp, double* sz, double* flops) {
    if (!d_psi) throw Err(ERR_ARG_WRONG, "psi is NULL.");
    if (!szsz || !spsm || !smsp || !sz) throw Err(ERR_ARG_WRONG, "an output matrix is NULL.");
    std::set<double> qns;
    for (const KronPair& p : kron->pairs) qns.insert(p.qn);
    if (qns.size() != 1)
        throw Err(ERR_SUP, "the correlation matrix needs a superblock of exactly one total-Sz sector (this one has " + std::to_string(qns.size()) + ").");
    const double qn = *qns.begin();
    Ctx* ctx = kron->ctx;
    const Block *L = kron->L, *R = kron->R;
    const int nL = L->nsites, nR = R->nsites, n = nL + nR;
    /* superblock site s: left-block site s, or right-block site nL + nR - 1 - s (hshell_create, SetUpCorrelation) */
    auto site_op = [&](int s, int type) { return s < nL ? L->op(type, s) : R->op(type, n - 1 - s); };
    for (int s = 0; s < n; ++s)
        if (!site_op(s, OP_SZ)->present || !site_op(s, OP_SP)->present)
            throw Err(ERR_ARG_WRONGSTATE, "superblock site " + std::to_string(s) + " (" + (s < nL ? "left" : "right") + " block site " +
                                              std::to_string(s < nL ? s : n - 1 - s) + "): Sz or Sp has not been set.");
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
            for (int s = 0; s < n; ++s) plan_panel(plan, kron, ok, s < nL, site_op(s, grp.type), d_psi, P + (long long)s * ldp);
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

}  // namespace dmrgx
