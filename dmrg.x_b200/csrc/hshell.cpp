/*  hshell.cpp — KronBlocks_t bookkeeping and the matrix-free superblock Hamiltonian
 *  (include/DMRGKron.hpp:117-480; src/DMRGKron.cpp:759-841, 891-989, 1706-1917).
 *
 *  The reference stores, per local row and per term, a 72-byte KronSumTermRow and pays nz_L·nz_R
 *  multiply-adds per row per term.  Here the same operator,
 *        Y_(IL,IR) += a · A[IL, IL+sA] · X_(IL+sA, IR+sB) · B[IR, IR+sB]ᵀ        (SURVEY.md §3.3)
 *  is planned once per superblock as two chain launches:
 *     stage 1   V_g,p = A_g[IL, IL+sA] · X_q                    one panel per distinct left operator g
 *     stage 2   Y_p   = Σ_g V_g,p · (Σ_j a_gj B_j[IR, IR+sB])ᵀ    all terms of a tile accumulated in registers
 *  Terms are grouped by their left operator; right operators of a group that share a panel shape are
 *  pre-summed at plan time.  Scaled-identity factors (H_L⊗1, 1⊗H_R, added-site operators) never
 *  generate a product: they alias X or turn into an in-register AXPY.
 */
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <set>

#include "common.h"
#include "plan.h"

namespace dmrgx {

/* include/DMRGKron.hpp:124-213 */
Kron* kron_create(const Block* L, const Block* R, const std::vector<double>& qn_sectors) {
    if (!L || !R) throw std::runtime_error("Left/right input block not initialized.");
    if (L->ctx != R->ctx) throw std::runtime_error("Left and right blocks must live in the same context.");
    std::unique_ptr<Kron> k(new Kron());
    k->ctx = L->ctx; k->L = L; k->R = R;
    const Sectors &SL = L->sec, &SR = R->sec;
    std::set<double> sel(qn_sectors.begin(), qn_sectors.end());
    for (int il = 0; il < SL.nsec(); ++il)
        for (int ir = 0; ir < SR.nsec(); ++ir) {
            const double qn = SL.qn[il] + SR.qn[ir];
            if (!qn_sectors.empty() && sel.find(qn) == sel.end()) continue; /* exact == on doubles, :165 */
            k->pairs.push_back({qn, il, ir, SL.size[il] * SR.size[ir]});
        }
    if (qn_sectors.empty()) /* only the keep-everything case is sorted (:157) */
        std::stable_sort(k->pairs.begin(), k->pairs.end(), [](const KronPair& a, const KronPair& b) { return a.qn > b.qn; });
    k->off.assign(k->pairs.size() + 1, 0);
    for (size_t p = 0; p < k->pairs.size(); ++p) {
        k->off[p + 1] = k->off[p] + k->pairs[p].size;
        k->map[{k->pairs[p].il, k->pairs[p].ir}] = (int)p;
    }
    return k.release();
}

namespace {
struct RightFactor { double coef; const Operator* B; };
struct Group {
    const Operator* A;      /* nullptr == identity */
    int sA, sB;
    std::vector<RightFactor> rights; /* B == nullptr == identity */
};
inline Tile full_eye(int off, int n) {
    Tile t;
    t.fmt = T_EYE; t.r0 = t.c0 = off; t.nr = t.nc = n; t.scale = 1.0;
    return t;
}
inline bool contiguous_dense(const Tile& t) {
    return t.fmt == T_DENSE && ((t.sc == 1 && t.sr == t.nc) || (t.sr == 1 && t.sc == t.nr));
}
}  // namespace

/* sub-tile made of rows [lo,hi) (global block coordinates) of a tile; false if empty */
static bool clip_tile_rows(Tile& t, int lo, int hi) {
    const int a = std::max(lo, t.r0), b = std::min(hi, t.r0 + t.nr);
    if (b <= a) return false;
    const int d = a - t.r0;
    if (t.fmt == T_DENSE) { t.d += (long long)d * t.sr; t.h_d0 += (long long)d * t.sr; }
    else if (t.fmt == T_CSR) { t.rowptr += d; t.h_rp += d; }   /* row pointers are absolute offsets into col/val */
    else { t.c0 += d; t.nc = b - a; }          /* a run of a scaled identity */
    t.r0 = a; t.nr = b - a;
    return true;
}

/* ------------------------------------------------------------------------------------------------
 *  Sparse-sector shell (north_star (a)).  When every operator tile the terms touch is CSR or a scaled identity — exact,
 *  un-truncated blocks handed over as CSR — the two-stage dense plan is replaced by one fused SpMM launch: per sector pair
 *  the terms Σ_t coef_t · A_t · X_q · B_tᵀ are evaluated row by row straight from ψ, with no V workspace at all
 *  (the reference's inner loop for these rows is src/DMRGKron.cpp:1844-1864).  The per-sector CSR of every factor is
 *  flattened on the host from the tiles' host copies (EYE runs become explicit entries) and uploaded once.
 * ---------------------------------------------------------------------------------------------- */
namespace {
struct FlatCsr { std::vector<int> rowptr, col; std::vector<double> val; long long ioff = 0, voff = 0; };

/* rows of sector I of operator O (columns local to sector J) as CSR; false when a tile has no host copy (device-born panels) */
bool flatten_sector(const Operator* O, const Sectors& S, int I, int J, FlatCsr& out) {
    const int nI = S.size[I];
    std::vector<std::vector<std::pair<int, double>>> rows(nI);
    for (const Tile& t : O->tiles[I]) {
        const int r0 = t.r0 - S.off[I], c0 = t.c0 - S.off[J];
        if (t.fmt == T_DENSE) {
            if (!t.hdense) return false;
            const std::vector<double>& h = *t.hdense;
            for (int i = 0; i < t.nr; ++i)
                for (int j = 0; j < t.nc; ++j) {
                    const double v = h[(size_t)(t.h_d0 + (long long)i * t.sr + (long long)j * t.sc)];
                    if (v != 0.0) rows[r0 + i].push_back({c0 + j, v});
                }
        } else if (t.fmt == T_EYE) {
            for (int i = 0; i < t.nr; ++i) rows[r0 + i].push_back({c0 + i, t.scale});
        } else {
            if (!t.hcsr) return false;
            const HostCsr& h = *t.hcsr;
            for (int i = 0; i < t.nr; ++i)
                for (int e = h.rowptr[t.h_rp + i]; e < h.rowptr[t.h_rp + i + 1]; ++e) rows[r0 + i].push_back({c0 + h.col[t.h_ci + e], h.val[t.h_ci + e]});
        }
    }
    out.rowptr.assign(nI + 1, 0);
    for (int i = 0; i < nI; ++i) {
        auto& r = rows[i];
        std::sort(r.begin(), r.end(), [](const std::pair<int, double>& a, const std::pair<int, double>& b) { return a.first < b.first; });
        for (size_t k = 0; k < r.size(); ++k) {
            if (k > 0 && r[k].first == out.col.back() && (int)out.col.size() > out.rowptr[i]) out.val.back() += r[k].second;
            else { out.col.push_back(r[k].first); out.val.push_back(r[k].second); }
        }
        out.rowptr[i + 1] = (int)out.col.size();
    }
    return true;
}
}  // namespace

/* Returns false (and leaves H untouched) when the superblock is not purely sparse. */
static bool try_build_sparse(HShell* H, const Kron* kron, const std::vector<Group>& groups, const std::vector<int>& lr0, const std::vector<int>& lr1,
                             long long& tile_bytes, bool dry) {
    if (getenv("DMRGX_NO_SPARSE")) return false; /* experiment / test hook: force the chain-kernel path */
    const bool force = getenv("DMRGX_FORCE_SPARSE") != nullptr; /* test hook: skip the fill criterion (general CSR factors with long rows) */
    Ctx* ctx = kron->ctx;
    const Sectors &SL = kron->L->sec, &SR = kron->R->sec;
    const int np = (int)kron->pairs.size();
    /* sparse means: every tile came from the host (CSR, identity runs, or one of the small filled blocks at the edge of an exact
       block) and the operators are sparse overall — stored non-zeros at most a quarter of the sector-block areas they live in */
    {
        double nnz = 0, area = 0;
        auto scan = [&](const Operator* O) {
            for (const auto& v : O->tiles)
                for (const Tile& t : v) {
                    if ((t.fmt == T_DENSE && !t.hdense) || (t.fmt == T_CSR && !t.hcsr)) return false;
                    nnz += t.fmt == T_DENSE ? (double)t.nr * t.nc : (t.fmt == T_CSR ? (double)t.nnz : (double)t.nr);
                    area += (double)t.nr * t.nc;
                }
            return true;
        };
        for (const Group& G : groups) {
            if (G.A && !scan(G.A)) return false;
            for (const RightFactor& rf : G.rights) if (rf.B && !scan(rf.B)) return false;
        }
        if (!force && area > 65536.0 && nnz > 0.25 * area) return false;
    }
    for (int p = 0; p < np; ++p) if (SR.size[kron->pairs[p].ir] > dev::SP_MAX_NR) return false;

    std::unique_ptr<SparsePlan> sp(new SparsePlan());
    /* flattened factors, cached per (operator, sector): left factors stay on the host (they are folded into the row programs),
       right factors become sliced-ELL device arrays */
    struct Ell { std::vector<int> col; std::vector<double> val; int W = 0, ld = 0; long long ioff = 0, voff = 0; };
    std::map<std::pair<const Operator*, int>, std::shared_ptr<FlatCsr>> cacheL;
    std::map<std::pair<const Operator*, int>, std::shared_ptr<Ell>> cacheR;
    std::vector<std::shared_ptr<Ell>> ells;
    auto getL = [&](const Operator* O, int I, int J) {
        auto key = std::make_pair(O, I);
        auto f = cacheL.find(key);
        if (f != cacheL.end()) return f->second;
        auto fc = std::make_shared<FlatCsr>();
        if (!flatten_sector(O, SL, I, J, *fc)) throw Err(ERR_GENERIC, "sparse shell: tile without a host copy");
        cacheL[key] = fc;
        return fc;
    };
    /* right factor as slot-major ELL over its rows (= the output columns): entry t of column c at [t*ld + c] */
    auto getR = [&](const Operator* O, int I, int J) {
        auto key = std::make_pair(O, I);
        auto f = cacheR.find(key);
        if (f != cacheR.end()) return f->second;
        FlatCsr fc;
        if (!flatten_sector(O, SR, I, J, fc)) throw Err(ERR_GENERIC, "sparse shell: tile without a host copy");
        auto el = std::make_shared<Ell>();
        const int n = SR.size[I];
        el->ld = (n + 31) & ~31;
        for (int c = 0; c < n; ++c) el->W = std::max(el->W, fc.rowptr[c + 1] - fc.rowptr[c]);
        el->col.assign((size_t)el->W * el->ld, 0);
        el->val.assign((size_t)el->W * el->ld, 0.0);
        for (int c = 0; c < n; ++c)
            for (int e = fc.rowptr[c], t = 0; e < fc.rowptr[c + 1]; ++e, ++t) { el->col[(size_t)t * el->ld + c] = fc.col[e]; el->val[(size_t)t * el->ld + c] = fc.val[e]; }
        cacheR[key] = el; ells.push_back(el);
        return el;
    };
    std::set<const void*> touched;
    auto touch = [&](const Tile& t) {
        const void* key = t.fmt == T_CSR ? (const void*)t.val : (t.fmt == T_DENSE ? (const void*)t.d : nullptr);
        if (key && touched.insert(key).second) tile_bytes += t.bytes();
    };
    std::vector<int> bslot_ell; /* right factor of every SpBSlot, by index, until the device arrays exist */
    for (int p = 0; p < np; ++p) {
        const int il = kron->pairs[p].il, ir = kron->pairs[p].ir;
        const int nR = SR.size[ir];
        if (lr1[p] <= lr0[p] || nR == 0) continue;
        sp->max_nR = std::max(sp->max_nR, nR);
        struct PT { std::shared_ptr<FlatCsr> a; int ell; long long xoff; int nRq; double coef; };
        std::vector<PT> pts;
        for (const Group& G : groups) {
            const int jl = il + G.sA, jr = ir + G.sB;
            if (jl < 0 || jl >= SL.nsec() || jr < 0 || jr >= SR.nsec()) continue;
            const int q = kron->find(jl, jr);
            if (q < 0 || SL.size[jl] == 0 || SR.size[jr] == 0) continue;
            std::shared_ptr<FlatCsr> a;
            if (G.A) { a = getL(G.A, il, jl); for (const Tile& t : G.A->tiles[il]) touch(t); }
            for (const RightFactor& rf : G.rights) {
                int ell = -1;
                double bnnz = nR;
                if (rf.B) {
                    auto el = getR(rf.B, ir, jr);
                    for (const Tile& t : rf.B->tiles[ir]) touch(t);
                    if (el->W == 0) continue;
                    ell = (int)(std::find(ells.begin(), ells.end(), el) - ells.begin());
                    bnnz = 0;
                    for (double v : el->val) bnnz += v != 0.0;
                }
                pts.push_back({a, ell, kron->off[q], SR.size[jr], rf.coef});
                const double annz = a ? (double)(a->rowptr[lr1[p]] - a->rowptr[lr0[p]]) : (double)(lr1[p] - lr0[p]);
                sp->flops += 2.0 * annz * bnnz;
            }
        }
        for (int l0 = lr0[p]; l0 < lr1[p]; l0 += dev::SP_ROWS) {
            dev::SpTile tl;
            std::memset(&tl, 0, sizeof tl);
            tl.nR = nR; tl.nrows = std::min(dev::SP_ROWS, lr1[p] - l0);
            tl.off = kron->off[p] + (long long)l0 * nR;
            /* the entries of row r in term t: (source row offset, weight) */
            auto row_entries = [&](const PT& t, int l, std::vector<std::pair<long long, double>>& out) {
                if (!t.a) { out.push_back({t.xoff + (long long)l * t.nRq, t.coef}); return; }
                for (int e = t.a->rowptr[l]; e < t.a->rowptr[l + 1]; ++e) out.push_back({t.xoff + (long long)t.a->col[e] * t.nRq, t.coef * t.a->val[e]});
            };
            /* identity-right entries of all terms, slot-major over the rows */
            std::vector<std::vector<std::pair<long long, double>>> al(dev::SP_ROWS);
            for (const PT& t : pts)
                if (t.ell < 0) for (int r = 0; r < tl.nrows; ++r) row_entries(t, l0 + r, al[r]);
            /* entries whose source row is one of the tile's own rows are served from shared memory: a list of their own */
            const long long t_end = tl.off + (long long)tl.nrows * nR;
            std::vector<std::vector<std::pair<long long, double>>> sl_(dev::SP_ROWS), gl_(dev::SP_ROWS);
            for (int r = 0; r < dev::SP_ROWS; ++r)
                for (auto& e : al[r]) (e.first >= tl.off && e.first < t_end ? sl_[r] : gl_[r]).push_back(e);
            size_t na = 0, ns = 0;
            for (auto& v : gl_) na = std::max(na, v.size());
            for (auto& v : sl_) ns = std::max(ns, v.size());
            tl.a_begin = (int)sp->aslots.size(); tl.a_count = (int)na;
            for (size_t k = 0; k < na; ++k) {
                dev::SpASlot sl;
                for (int r = 0; r < dev::SP_ROWS; ++r) {
                    const bool has = k < gl_[r].size();
                    sl.src[r] = has ? gl_[r][k].first : tl.off; sl.w[r] = has ? gl_[r][k].second : 0.0;
                }
                sp->aslots.push_back(sl);
            }
            tl.s_begin = (int)sp->sslots.size(); tl.s_count = (int)ns;
            for (size_t k = 0; k < ns; ++k) {
                dev::SpSSlot sl;
                std::memset(&sl, 0, sizeof sl);
                for (int r = 0; r < dev::SP_ROWS; ++r) {
                    const bool has = k < sl_[r].size();
                    sl.roff[r] = has ? (int)(sl_[r][k].first - tl.off) : 0; sl.w[r] = has ? sl_[r][k].second : 0.0;
                }
                sp->sslots.push_back(sl);
            }
            /* gather slots: (term, k-th left entry of each row) */
            tl.b_begin = (int)sp->bslots.size();
            for (const PT& t : pts) {
                if (t.ell < 0) continue;
                std::vector<std::vector<std::pair<long long, double>>> bl(dev::SP_ROWS);
                size_t nk = 0;
                for (int r = 0; r < tl.nrows; ++r) { row_entries(t, l0 + r, bl[r]); nk = std::max(nk, bl[r].size()); }
                for (size_t k = 0; k < nk; ++k) {
                    dev::SpBSlot sl;
                    std::memset(&sl, 0, sizeof sl);
                    sl.W = ells[(size_t)t.ell]->W; sl.ld = ells[(size_t)t.ell]->ld;
                    sl.all_in = 1;
                    for (int r = 0; r < dev::SP_ROWS; ++r) {
                        const bool has = k < bl[r].size();
                        sl.src[r] = has ? bl[r][k].first : tl.off; sl.w[r] = has ? bl[r][k].second : 0.0;
                        const bool in = sl.src[r] >= tl.off && sl.src[r] < tl.off + (long long)tl.nrows * nR;
                        sl.roff[r] = in ? (int)(sl.src[r] - tl.off) : 0;
                        sl.all_in &= in ? 1 : 0;
                    }
                    sp->bslots.push_back(sl);
                    bslot_ell.push_back(t.ell);
                }
            }
            tl.b_count = (int)sp->bslots.size() - tl.b_begin;
            sp->tiles.push_back(tl);
        }
    }
    /* widest rows first: the hardware dispatches CTAs in index order (LPT) */
    std::stable_sort(sp->tiles.begin(), sp->tiles.end(), [](const dev::SpTile& a, const dev::SpTile& b) { return a.nR > b.nR; });
    if (!dry) {
        long long ni = 0, nv = 0;
        for (auto& el : ells) { el->ioff = ni; ni += (long long)el->col.size(); el->voff = nv; nv += (long long)el->val.size(); }
        std::vector<int> hi((size_t)std::max<long long>(1, ni));
        std::vector<double> hv((size_t)std::max<long long>(1, nv));
        for (auto& el : ells) {
            std::copy(el->col.begin(), el->col.end(), hi.begin() + el->ioff);
            std::copy(el->val.begin(), el->val.end(), hv.begin() + el->voff);
        }
        sp->d_int = std::make_shared<DevBuf>(ctx, hi.size() * 4);
        sp->d_val = std::make_shared<DevBuf>(ctx, hv.size() * 8);
        dev::h2d(ctx->st, sp->d_int->p, hi.data(), hi.size() * 4);
        dev::h2d(ctx->st, sp->d_val->p, hv.data(), hv.size() * 8);
        for (size_t i = 0; i < sp->bslots.size(); ++i) {
            const Ell& el = *ells[(size_t)bslot_ell[i]];
            sp->bslots[i].ecol = sp->d_int->as<int>() + el.ioff;
            sp->bslots[i].eval = sp->d_val->as<double>() + el.voff;
        }
        sp->d_tiles = std::make_shared<DevBuf>(ctx, std::max<size_t>(1, sp->tiles.size()) * sizeof(dev::SpTile));
        sp->d_aslots = std::make_shared<DevBuf>(ctx, std::max<size_t>(1, sp->aslots.size()) * sizeof(dev::SpASlot));
        sp->d_sslots = std::make_shared<DevBuf>(ctx, std::max<size_t>(1, sp->sslots.size()) * sizeof(dev::SpSSlot));
        dev::h2d(ctx->st, sp->d_sslots->p, sp->sslots.data(), sp->sslots.size() * sizeof(dev::SpSSlot));
        sp->d_bslots = std::make_shared<DevBuf>(ctx, std::max<size_t>(1, sp->bslots.size()) * sizeof(dev::SpBSlot));
        dev::h2d(ctx->st, sp->d_tiles->p, sp->tiles.data(), sp->tiles.size() * sizeof(dev::SpTile));
        dev::h2d(ctx->st, sp->d_aslots->p, sp->aslots.data(), sp->aslots.size() * sizeof(dev::SpASlot));
        dev::h2d(ctx->st, sp->d_bslots->p, sp->bslots.data(), sp->bslots.size() * sizeof(dev::SpBSlot));
        dev::sync(ctx->st);
    }
    H->sparse = std::move(sp);
    return true;
}

/* Builds the two-stage plan of the shell.  [row_begin,row_end) is the range of superblock rows this rank owns (cut at
   left-row boundaries of the sector pairs; the whole vector on one GPU): only those rows of V and Y are planned, so the
   ranks partition the work exactly, with no redundant products (the successor of KronSumShellSplitOwnership,
   src/DMRGKron.cpp:1519-1704).  dry = cost model only: nothing is allocated, summed or uploaded; pair_cost receives the
   useful flops per sector pair. */
static HShell* build_shell(const Kron* kron, const std::vector<Group>& groups, int nterms, long long row_begin = 0, long long row_end = -1,
                           bool dry = false, std::vector<double>* pair_cost = nullptr) {
    Ctx* ctx = kron->ctx;
    Trace tr(ctx, dry ? "build_shell(dry)" : "build_shell");
    std::unique_ptr<HShell> H(new HShell());
    H->ctx = ctx; H->kron = kron; H->n = kron->nstates(); H->nterms = nterms;
    if (row_end < 0) row_end = H->n;
    H->row_begin = row_begin; H->row_end = row_end;
    const Sectors &SL = kron->L->sec, &SR = kron->R->sec;
    const int np = (int)kron->pairs.size();
    /* owned left rows [lr0,lr1) of every pair */
    std::vector<int> lr0(np, 0), lr1(np, 0);
    for (int p = 0; p < np; ++p) {
        const long long nR = SR.size[kron->pairs[p].ir];
        if (nR == 0) continue;
        const long long a = std::max(row_begin, kron->off[p]) - kron->off[p], b = std::min(row_end, kron->off[p + 1]) - kron->off[p];
        if (b <= a) continue;
        if (a % nR || b % nR) throw Err(ERR_GENERIC, "row ownership must be cut at left-row boundaries of the sector pairs");
        lr0[p] = (int)(a / nR); lr1[p] = (int)(b / nR);
    }
    if (pair_cost) pair_cost->assign(np, 0.0);
    std::set<const void*> touched;
    long long tile_bytes = 0;
    auto touch = [&](const Tile& t) {
        const void* key = t.fmt == T_DENSE ? (const void*)t.d : (t.fmt == T_CSR ? (const void*)t.val : nullptr);
        if (key && touched.insert(key).second) tile_bytes += t.bytes();
    };

    /* ---- purely sparse superblock (exact blocks handed over as CSR): one fused SpMM launch instead of the two-stage plan ---- */
    if (try_build_sparse(H.get(), kron, groups, lr0, lr1, tile_bytes, dry)) {
        if (pair_cost) {
            for (int p = 0; p < np; ++p) (*pair_cost)[p] = (double)(lr1[p] - lr0[p]) * SR.size[kron->pairs[p].ir];
        }
        H->alg_bytes = 16LL * H->n + tile_bytes;
        H->alg_flops = H->sparse->flops;
        tr.mark("sparse plan");
        return H.release();
    }

    /* ---- pass 1: size the V workspace ---- */
    struct GP { long long voff; int q; };
    std::vector<std::vector<GP>> gp(groups.size(), std::vector<GP>(np, GP{-1, -1}));
    long long wtotal = 0;
    for (size_t g = 0; g < groups.size(); ++g) {
        const Group& G = groups[g];
        for (int p = 0; p < np; ++p) {
            const int il = kron->pairs[p].il, ir = kron->pairs[p].ir;
            const int jl = il + G.sA, jr = ir + G.sB;
            if (jl < 0 || jl >= SL.nsec() || jr < 0 || jr >= SR.nsec()) continue;
            const int q = kron->find(jl, jr);
            if (q < 0) continue;
            gp[g][p].q = q;
            bool needV = false;
            if (G.A)
                for (const Tile& t : G.A->tiles[il]) if (t.fmt != T_EYE) needV = true;
            if (lr1[p] <= lr0[p]) { gp[g][p].q = -1; continue; }
            if (needV) { gp[g][p].voff = wtotal; wtotal += (long long)(lr1[p] - lr0[p]) * SR.size[jr]; }
        }
    }
    if (!dry) H->work = std::make_shared<DevBuf>(ctx, std::max<long long>(1, wtotal) * 8);
    double* W = dry ? nullptr : H->work->as<double>();

    /* ---- pre-summed right factors per (group, right row sector) ---- */
    struct BTile { Tile t; double coef; };
    std::vector<std::vector<std::vector<BTile>>> bt(groups.size(), std::vector<std::vector<BTile>>(SR.nsec()));
    /* An operator of the enlarged block is O_i ⊗ 1_site: the SAME panel is referenced from two enlarged sectors (site up / site
       down).  Sums over the same source panels with the same coefficients are therefore materialised once and shared
       (halves the derived panels: 185 -> 93 MB at 12x6 m = 2048, less DRAM traffic and L2 pressure in stage 2). */
    std::map<std::vector<std::pair<const double*, double>>, BufRef> sum_cache;
    for (size_t g = 0; g < groups.size(); ++g) {
        const Group& G = groups[g];
        for (int ir = 0; ir < SR.nsec(); ++ir) {
            const int jr = ir + G.sB;
            if (jr < 0 || jr >= SR.nsec()) continue;
            std::vector<BTile> raw;
            for (const RightFactor& rf : G.rights) {
                if (!rf.B) { if (SR.size[ir] > 0) raw.push_back({full_eye(SR.off[ir], SR.size[ir]), rf.coef}); continue; }
                for (const Tile& t : rf.B->tiles[ir]) raw.push_back({t, rf.coef});
            }
            std::vector<char> used(raw.size(), 0);
            for (size_t a = 0; a < raw.size(); ++a) {
                if (used[a]) continue;
                used[a] = 1;
                std::vector<size_t> same = {a};
                if (contiguous_dense(raw[a].t))
                    for (size_t b = a + 1; b < raw.size(); ++b)
                        if (!used[b] && contiguous_dense(raw[b].t) && raw[b].t.r0 == raw[a].t.r0 && raw[b].t.c0 == raw[a].t.c0 &&
                            raw[b].t.nr == raw[a].t.nr && raw[b].t.nc == raw[a].t.nc && raw[b].t.sr == raw[a].t.sr && raw[b].t.sc == raw[a].t.sc) {
                            same.push_back(b); used[b] = 1;
                        }
                /* a lone factor is used in place unless it carries a coefficient: the GEMM inner loop is free of
                   multiplies only for unit coefficients, so a·B is materialised too (one small axpy at plan time) */
                if (same.size() == 1 && (raw[a].coef == 1.0 || !contiguous_dense(raw[a].t))) { bt[g][ir].push_back(raw[a]); touch(raw[a].t); continue; }
                /* Σ_j a_j B_j materialised once (device axpy over the contiguous panels) */
                const long long cnt = (long long)raw[a].t.nr * raw[a].t.nc;
                BTile merged = raw[a];
                if (!dry) {
                    std::vector<std::pair<const double*, double>> key;
                    for (size_t k = 0; k < same.size(); ++k) key.push_back({raw[same[k]].t.d, raw[same[k]].coef});
                    std::sort(key.begin(), key.end());
                    BufRef& sum = sum_cache[key];
                    if (!sum) {
                        sum = std::make_shared<DevBuf>(ctx, cnt * 8);
                        for (size_t k = 0; k < key.size(); ++k)
                            dev::axpby_out(ctx->st, k == 0 ? nullptr : sum->as<double>(), key[k].first, key[k].second, sum->as<double>(), cnt);
                        H->keep.push_back(sum);
                    }
                    merged.t.d = sum->as<double>(); merged.t.owner = sum;
                }
                merged.coef = 1.0;
                bt[g][ir].push_back(merged);
                for (size_t k = 0; k < same.size(); ++k) touch(raw[same[k]].t); /* algorithmic bytes count the ORIGINAL panels once each */
            }
        }
    }

    tr.mark("presum");
    /* ---- stage 1: V panels;  stage 2: Y panels ---- */
    std::vector<std::vector<Contribution>> ycontrib(np);
    for (size_t g = 0; g < groups.size(); ++g) {
        const Group& G = groups[g];
        for (int p = 0; p < np; ++p) {
            const int q = gp[g][p].q;
            if (q < 0) continue;
            const int il = kron->pairs[p].il, ir = kron->pairs[p].ir;
            const int jl = il + G.sA, jr = ir + G.sB;
            const int nLp = lr1[p] - lr0[p], nRq = SR.size[jr];
            if (nLp <= 0 || SR.size[ir] == 0 || nRq == 0 || SL.size[jl] == 0) continue;
            const long long xq = kron->off[q];
            std::vector<Tile> atiles;
            if (G.A) atiles = G.A->tiles[il]; else atiles.push_back(full_eye(SL.off[il], SL.size[il]));
            std::vector<Contribution> vcontrib;
            const double flops_before = H->stage1.flops;
            for (Tile a : atiles) {
                if (!clip_tile_rows(a, SL.off[il] + lr0[p], SL.off[il] + lr1[p])) continue;
                /* rows are counted from the first owned row of the pair */
                const int ra0 = a.r0 - SL.off[il] - lr0[p], ca0 = a.c0 - SL.off[jl];
                /* --- the left factor --- */
                const double* vsrc; int vflags; double acoef = 1.0;
                if (a.fmt == T_EYE) {
                    vsrc = xoff(xq + (long long)ca0 * nRq); vflags = dev::SEGF_A_X; acoef = a.scale;
                } else {
                    touch(a);
                    vsrc = W + gp[g][p].voff + (long long)ra0 * nRq; vflags = 0;
                    Contribution c;
                    c.r0 = ra0; c.c0 = 0; c.nr = a.nr; c.nc = nRq;
                    if (a.fmt == T_DENSE) {
                        c.seg = make_seg(dev::SEG_GEMM);
                        c.seg.A = a.d; c.seg.lda_m = a.sr; c.seg.lda_k = a.sc; c.seg.K = a.nc;
                        c.seg.B = xoff(xq + (long long)ca0 * nRq); c.seg.ldb_k = nRq; c.seg.ldb_n = 1; c.seg.flags = dev::SEGF_B_X;
                    } else {
                        c.seg = make_seg(dev::SEG_CSRA);
                        c.seg.rowptr = a.rowptr; c.seg.colidx = a.col; c.seg.B = a.val;
                        c.seg.A = xoff(xq + (long long)ca0 * nRq); c.seg.ldb_k = nRq; c.seg.ldb_n = 1; c.seg.flags = dev::SEGF_A_X;
                    }
                    vcontrib.push_back(c);
                }
                /* --- times every right factor of the group --- */
                for (const BTile& bb : bt[g][ir]) {
                    const Tile& b = bb.t;
                    const int rb0 = b.r0 - SR.off[ir], cb0 = b.c0 - SR.off[jr];
                    Contribution c;
                    c.r0 = ra0; c.nr = a.nr; c.c0 = rb0; c.nc = b.nr;
                    if (b.fmt == T_DENSE) {
                        c.seg = make_seg(dev::SEG_GEMM);
                        c.seg.A = vsrc + cb0; c.seg.lda_m = nRq; c.seg.lda_k = 1; c.seg.K = b.nc;
                        c.seg.B = b.d; c.seg.ldb_n = b.sr; c.seg.ldb_k = b.sc;
                        c.seg.coef = acoef * bb.coef;
                    } else if (b.fmt == T_EYE) {
                        c.seg = make_seg(dev::SEG_AXPY);
                        c.seg.A = vsrc + cb0; c.seg.lda_m = nRq; c.seg.lda_k = 1;
                        c.seg.coef = acoef * bb.coef * b.scale;
                    } else {
                        c.seg = make_seg(dev::SEG_CSRB);
                        c.seg.A = vsrc + cb0; c.seg.lda_m = nRq; c.seg.lda_k = 1;
                        c.seg.rowptr = b.rowptr; c.seg.colidx = b.col; c.seg.B = b.val;
                        c.seg.coef = acoef * bb.coef;
                    }
                    c.seg.flags |= vflags;
                    ycontrib[p].push_back(c);
                }
            }
            if (!vcontrib.empty()) emit_cells(H->stage1, W + gp[g][p].voff, false, nRq, nLp, nRq, vcontrib, false);
            if (pair_cost) (*pair_cost)[p] += H->stage1.flops - flops_before;
        }
    }
    {   /* dry run to learn the total stage-2 work, then cut long chains so that the launch has about two waves of
           equal items on 148 SMs x 3 resident CTAs (v0 lost a third of the machine to a 1.4-wave tail) */
        Plan probe;
        for (int p = 0; p < np; ++p)
            emit_cells(probe, yoff(kron->off[p]), true, SR.size[kron->pairs[p].ir], lr1[p] - lr0[p], SR.size[kron->pairs[p].ir], ycontrib[p], true);
        /* How many work items the launch should have: one wave of the 444 resident CTAs for light superblocks, up to three for
           heavy ones (about one item per 40 full-tile chunks of work).  Parts of a cut chain go through the scratch buffer and
           the reduce pass, so more parts than needed to even out the last wave only add traffic: measured optima were 574 items
           at m = 512, 858 at m = 1024 and 2012 at m = 2048 (profiles/r1_chain_kernel.md). */
        const double chunks_total = probe.flops / (2.0 * 64 * 64 * 16);
        const double target_items = std::min(3.0 * 444.0, std::max(444.0, chunks_total / 40.0));
        if (probe.flops > 0 && (double)probe.items.size() < target_items) H->stage2.split_item_cost = 0.5 * probe.flops / target_items;
    }
    for (int p = 0; p < np; ++p) {
        const int nLp = lr1[p] - lr0[p], nRp = SR.size[kron->pairs[p].ir];
        const double flops_before = H->stage2.flops;
        /* y offsets are global: a rank that stores only its own rows passes y - row_begin as the base */
        emit_cells(H->stage2, yoff(kron->off[p] + (long long)lr0[p] * nRp), true, nRp, nLp, nRp, ycontrib[p], true);
        if (pair_cost) (*pair_cost)[p] += H->stage2.flops - flops_before;
    }
    tr.mark("plan");
    if (!dry) {
        H->stage1.upload(ctx);
        H->stage2.upload(ctx);
    }
    tr.mark("upload");
    H->alg_bytes = 16LL * H->n + tile_bytes;
    H->alg_flops = H->stage1.flops + H->stage2.flops;
    return H.release();
}

/* Row ownership of the ranks (a5, src/DMRGKron.cpp:1519-1704: contiguous row ranges with even predicted work; falls back
   to an even split of rows when there is nothing to predict).  The prediction is the plan's own useful flops per sector
   pair, spread evenly over the pair's left rows; cuts fall on left-row boundaries, on multiples of 16 rows where the pair
   is large enough (whole DMMA fragments).  Every rank computes the same table. */
static std::vector<long long> shard_rows(const Kron* kron, const std::vector<Group>& groups, int nterms, int world, long long& global_bytes,
                                         double& global_flops) {
    const int np = (int)kron->pairs.size();
    const long long n = kron->nstates();
    std::vector<long long> cuts(world + 1, n);
    cuts[0] = 0;
    if (world <= 1) return cuts;
    std::vector<double> cost;
    { std::unique_ptr<HShell> probe(build_shell(kron, groups, nterms, 0, -1, true, &cost)); global_bytes = probe->alg_bytes; global_flops = probe->alg_flops; }
    const Sectors &SL = kron->L->sec, &SR = kron->R->sec;
    double total = 0;
    for (int p = 0; p < np; ++p) {
        if (cost[p] <= 0) cost[p] = (double)kron->pairs[p].size; /* sparse / identity-only pairs: count rows */
        total += cost[p];
    }
    if (total <= 0) { for (int r = 1; r < world; ++r) cuts[r] = 0; return cuts; }
    double cum = 0;
    int r = 1;
    for (int p = 0; p < np && r < world; ++p) {
        const long long nL = SL.size[kron->pairs[p].il], nR = SR.size[kron->pairs[p].ir];
        while (r < world && cost[p] > 0 && total * r / world <= cum + cost[p]) {
            const double frac = (total * r / world - cum) / cost[p];
            long long l = (long long)std::llround(frac * (double)nL);
            if (nL >= 64) l = ((l + 8) / 16) * 16;
            l = std::max<long long>(0, std::min(l, nL));
            cuts[r] = std::max(cuts[r - 1], kron->off[p] + l * nR);
            ++r;
        }
        cum += cost[p];
    }
    for (; r < world; ++r) cuts[r] = n;
    return cuts;
}

/* The sector halo (SURVEY.md §8e; the reference gathers ALL of psi on every rank, src/DMRGKron.cpp:1833-1834): a rank's tiles read
   only the pairs q = (IL + sA, IR + sB) of its own pairs' terms — Sz shifts of -1, 0, +1, i.e. neighbouring sector pairs.
   Every rank derives the needs of every rank from the ownership table, so all ranks hold the same transfer list. */
static void plan_halo(HShell* H, const Kron* kron, const std::vector<Group>& groups, const std::vector<long long>& cuts) {
    const Sectors &SL = kron->L->sec, &SR = kron->R->sec;
    const int np = (int)kron->pairs.size(), world = (int)cuts.size() - 1, me = kron->ctx->rank;
    for (int r = 0; r < world; ++r) {
        std::vector<char> need(np, 0);
        for (int p = 0; p < np; ++p) {
            if (std::min(cuts[r + 1], kron->off[p + 1]) <= std::max(cuts[r], kron->off[p])) continue; /* rank r owns no row of pair p */
            for (const Group& G : groups) {
                const int jl = kron->pairs[p].il + G.sA, jr = kron->pairs[p].ir + G.sB;
                if (jl < 0 || jl >= SL.nsec() || jr < 0 || jr >= SR.nsec()) continue;
                const int q = kron->find(jl, jr);
                if (q >= 0 && G.A) need[q] = 1; /* an identity left factor reads the rank's own rows only */
            }
        }
        for (int q = 0; q < np; ++q) {
            if (!need[q]) continue;
            for (int s = 0; s < world; ++s) {
                if (s == r) continue;
                const long long a = std::max(kron->off[q], cuts[s]), b = std::min(kron->off[q + 1], cuts[s + 1]);
                if (b <= a) continue;
                /* merge with the previous transfer of the same (s, r) when contiguous */
                if (!H->halo_from.empty() && H->halo_from.back() == s && H->halo_to.back() == r && H->halo_off.back() + H->halo_cnt.back() == a) H->halo_cnt.back() += b - a;
                else { H->halo_from.push_back(s); H->halo_to.push_back(r); H->halo_off.push_back(a); H->halo_cnt.push_back(b - a); }
            }
        }
    }
    for (size_t i = 0; i < H->halo_to.size(); ++i) if (H->halo_to[i] == me) H->halo_recv_elems += H->halo_cnt[i];
}

static HShell* build_sharded(const Kron* kron, const std::vector<Group>& groups, int nterms) {
    Ctx* ctx = kron->ctx;
    if (ctx->world <= 1) {
        HShell* H = build_shell(kron, groups, nterms);
        H->row_cuts = {0, H->n};
        H->alg_bytes_global = H->alg_bytes; H->alg_flops_global = H->alg_flops;
        return H;
    }
    long long gb = 0; double gf = 0;
    const std::vector<long long> cuts = shard_rows(kron, groups, nterms, ctx->world, gb, gf);
    HShell* H = build_shell(kron, groups, nterms, cuts[ctx->rank], cuts[ctx->rank + 1]);
    H->row_cuts = cuts;
    H->alg_bytes_global = gb; H->alg_flops_global = gf;
    plan_halo(H, kron, groups, cuts);
    return H;
}

/* src/DMRGKron.cpp:759-841 (classification, reflection) + :891-989 (term list = H_L⊗1, 1⊗H_R, LR terms) */
HShell* hshell_create(const Kron* kron, const std::vector<Term>& terms) {
    const Block *L = kron->L, *R = kron->R;
    const int nsL = L->nsites, nsR = R->nsites, nsO = nsL + nsR;
    long long maxsite = 0;
    for (const Term& t : terms) maxsite = std::max({maxsite, t.Isite, t.Jsite});
    if (maxsite >= nsO) throw Err(ERR_GENERIC, "Maximum site index from Terms has to be less than the total number of sites in the blocks.");
    block_check(L);
    block_check(R);
    std::vector<Term> lr;
    for (const Term& t : terms) {
        if (t.Isite >= 0 && t.Isite < nsL && t.Jsite >= nsL && t.Jsite < nsO) {
            if (t.a == 0.0) continue;
            Term u = t;
            u.Jsite = nsO - 1 - t.Jsite;
            lr.push_back(u);
        } else if (t.Isite >= 0 && t.Isite < nsL && t.Jsite >= 0 && t.Jsite < nsL) {
        } else if (t.Isite >= nsL && t.Isite < nsO && t.Jsite >= nsL && t.Jsite < nsO) {
        } else throw Err(ERR_GENERIC, "Invalid term.");
    }
    std::vector<Group> groups;
    groups.push_back({&L->H, 0, 0, {{1.0, nullptr}}});  /* H_L ⊗ 1 */
    groups.push_back({nullptr, 0, 0, {{1.0, &R->H}}});  /* 1 ⊗ H_R */
    std::map<std::tuple<int, long long, int>, size_t> gidx;
    for (const Term& t : lr) {
        if (t.Iop < OP_SM || t.Iop > OP_SP || t.Jop < OP_SM || t.Jop > OP_SP) throw Err(ERR_ARG_WRONG, "Incorrect operator type.");
        const Operator* A = L->op(t.Iop, (int)t.Isite);
        const Operator* B = R->op(t.Jop, (int)t.Jsite);
        auto key = std::make_tuple(t.Iop, t.Isite, t.Jop);
        auto f = gidx.find(key);
        if (f == gidx.end()) { gidx[key] = groups.size(); groups.push_back({A, t.Iop, t.Jop, {}}); f = gidx.find(key); }
        groups[f->second].rights.push_back({t.a, B});
    }
    return build_sharded(kron, groups, 2 + (int)lr.size());
}

/* KronConstruct, include/DMRGKron.hpp:309 / src/DMRGKron.cpp:618-694: one term 1.0 · A ⊗ B (correlators) */
HShell* hshell_create_single(const Kron* kron, int opl, int il, int opr, int ir) {
    const Operator* A = opl == OP_EYE ? nullptr : kron->L->op(opl, il);
    const Operator* B = opr == OP_EYE ? nullptr : kron->R->op(opr, ir);
    std::vector<Group> groups;
    groups.push_back({A, opl == OP_EYE ? 0 : opl, opr == OP_EYE ? 0 : opr, {{1.0, B}}});
    return build_sharded(kron, groups, 1);
}

/* Product O_1·O_2·…·O_k of operators of ONE block (CalculateOperatorProducts, include/DMRGBlockContainer.hpp:2340-2425:
   MatMatMult chain in list order), built right to left on the device as dense sector panels: any tile format may
   stand on the left (dense -> DMMA GEMM, CSR -> CSRA, scaled identity -> AXPY) of the dense running product. */
static std::shared_ptr<Operator> operator_product(const Block* blk, const std::vector<std::pair<int, int>>& ops, std::vector<BufRef>& keep) {
    Ctx* ctx = blk->ctx;
    const Sectors& S = blk->sec;
    const int ns = S.nsec();
    std::shared_ptr<Operator> P;
    for (int k = (int)ops.size() - 1; k >= 0; --k) {
        const Operator* O = blk->op(ops[k].first, ops[k].second);
        std::shared_ptr<Operator> N = std::make_shared<Operator>();
        N->shift = O->shift + (P ? P->shift : 0);
        N->present = true;
        N->tiles.assign(ns, {});
        std::vector<long long> off(ns + 1, 0);
        for (int I = 0; I < ns; ++I) {
            const int J = I + N->shift;
            off[I + 1] = off[I] + ((J >= 0 && J < ns) ? (long long)S.size[I] * S.size[J] : 0);
        }
        BufRef buf = std::make_shared<DevBuf>(ctx, std::max<long long>(1, off[ns]) * 8);
        keep.push_back(buf);
        Plan plan;
        for (int I = 0; I < ns; ++I) {
            const int J = I + N->shift, M = I + O->shift; /* O: I -> M, P: M -> J */
            if (J < 0 || J >= ns || S.size[I] == 0 || S.size[J] == 0) continue;
            double* out = buf->as<double>() + off[I];
            const int nI = S.size[I], nJ = S.size[J];
            std::vector<Contribution> cs;
            if (M >= 0 && M < ns) {
                for (const Tile& a : O->tiles[I]) {
                    const int ra0 = a.r0 - S.off[I], ca0 = a.c0 - S.off[M];
                    if (!P) { cs.push_back(add_tile_contribution(a, ra0, ca0, 1.0)); continue; }
                    for (const Tile& b : P->tiles[M]) { /* one dense panel covering the whole (M,J) block */
                        Contribution c;
                        c.r0 = ra0; c.c0 = 0; c.nr = a.nr; c.nc = nJ;
                        const double* bsrc = b.d + (long long)ca0 * nJ;
                        if (a.fmt == T_DENSE) {
                            c.seg = make_seg(dev::SEG_GEMM);
                            c.seg.A = a.d; c.seg.lda_m = a.sr; c.seg.lda_k = a.sc; c.seg.K = a.nc;
                            c.seg.B = bsrc; c.seg.ldb_k = nJ; c.seg.ldb_n = 1;
                        } else if (a.fmt == T_EYE) {
                            c.seg = make_seg(dev::SEG_AXPY);
                            c.seg.A = bsrc; c.seg.lda_m = nJ; c.seg.lda_k = 1; c.seg.coef = a.scale;
                        } else {
                            c.seg = make_seg(dev::SEG_CSRA);
                            c.seg.rowptr = a.rowptr; c.seg.colidx = a.col; c.seg.B = a.val;
                            c.seg.A = bsrc; c.seg.ldb_k = nJ; c.seg.ldb_n = 1;
                        }
                        cs.push_back(c);
                    }
                }
            }
            emit_cells(plan, out, false, nJ, nI, nJ, cs, true);
            Tile t;
            t.fmt = T_DENSE; t.r0 = S.off[I]; t.c0 = S.off[J]; t.nr = nI; t.nc = nJ; t.d = out; t.sr = nJ; t.sc = 1; t.owner = buf;
            N->tiles[I].push_back(t);
        }
        plan.upload(ctx);
        plan.run(ctx);
        dev::sync(ctx->st); /* the plan's device lists die with this scope */
        P = N;
    }
    return P;
}

/* correlator shell: 1.0 · (Π SysOps) ⊗ (Π EnvOps), include/DMRGBlockContainer.hpp:2262-2296.  An empty list is the
   identity; a single operator is used in place; longer lists are multiplied out on the device first. */
HShell* hshell_create_product(const Kron* kron, const std::vector<std::pair<int, int>>& lops, const std::vector<std::pair<int, int>>& rops) {
    std::vector<BufRef> keep;
    std::vector<std::shared_ptr<Operator>> keep_ops;
    auto factor = [&](const Block* blk, const std::vector<std::pair<int, int>>& ops, int& shift) -> const Operator* {
        shift = 0;
        for (auto& o : ops) {
            if (o.first < OP_SM || o.first > OP_SP) throw Err(ERR_ARG_WRONG, "Incorrect operator type.");
            shift += o.first;
        }
        if (ops.empty()) return nullptr;
        if (ops.size() == 1) return blk->op(ops[0].first, ops[0].second);
        keep_ops.push_back(operator_product(blk, ops, keep));
        return keep_ops.back().get();
    };
    int sA = 0, sB = 0;
    const Operator* A = factor(kron->L, lops, sA);
    const Operator* B = factor(kron->R, rops, sB);
    std::vector<Group> groups;
    groups.push_back({A, sA, sB, {{1.0, B}}});
    HShell* H = build_sharded(kron, groups, 1);
    H->keep.insert(H->keep.end(), keep.begin(), keep.end());
    H->keep_ops = keep_ops;
    return H;
}

/* MatMult_KronSumShell, src/DMRGKron.cpp:1827-1869 */
void hshell_apply(HShell* H, const double* d_x, double* d_y) {
    if (H->sparse) {
        const SparsePlan& sp = *H->sparse;
        dev::run_spmm(H->ctx->st, sp.d_tiles->as<dev::SpTile>(), (int)sp.tiles.size(), sp.d_aslots->as<dev::SpASlot>(), sp.d_sslots->as<dev::SpSSlot>(), sp.d_bslots->as<dev::SpBSlot>(), d_x, d_y,
                      sp.max_nR);
        return;
    }
    H->stage1.run(H->ctx, d_x, nullptr);
    H->stage2.run(H->ctx, d_x, d_y);
}

/* The distributed form of the callback: x is a full-length buffer in which only this rank's rows are valid on entry;
   the exchange step of the path (the VecScatter-to-all of src/DMRGKron.cpp:1833-1834) is the sector-halo exchange over
   NVLink, which brings this rank the rows of x its tiles read (plan_halo); then this rank computes its own rows of y. */
void hshell_apply_sharded(HShell* H, double* d_x, double* d_y) {
    if (H->ctx->world > 1)
        dev::exchange_ranges(H->ctx->st, d_x, (int)H->halo_from.size(), H->halo_from.data(), H->halo_to.data(), H->halo_off.data(), H->halo_cnt.data());
    hshell_apply(H, d_x, d_y);
}

}  // namespace dmrgx
