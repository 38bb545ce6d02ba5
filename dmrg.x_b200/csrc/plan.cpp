/*  plan.cpp — turns "output panel + list of rectangular contributions" into the flat work-item /
 *  segment lists the chain kernel consumes (dev.h).  Every output element is produced by exactly one
 *  work item, so there is no zero-fill pass and no atomics: the panel is cut along the edges of all
 *  contributing rectangles into cells, every cell is covered by a fixed set of contributions, and each
 *  cell is tiled with (almost) equal tiles of at most dev::TILE × dev::TILE.
 */
#include <algorithm>
#include <cmath>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.h"
#include "plan.h"

namespace dmrgx {

bool Trace::enabled() { static const bool on = getenv("DMRGX_TRACE") != nullptr; return on; }
double Trace::now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
Trace::Trace(Ctx* c, const char* w) : ctx(c), what(w), t0(0), on(enabled()) { if (on) { dev::sync(ctx->st); t0 = now(); } }
void Trace::mark(const char* label) {
    if (!on) return;
    dev::sync(ctx->st);
    const double t = now();
    fprintf(stderr, "[trace] %s.%s %.3f ms\n", what, label, (t - t0) * 1e3);
    t0 = t;
}

void Plan::upload(Ctx* ctx) {
    if (items.empty()) return;
    /* heaviest tiles first: the hardware dispatches CTAs in index order, so this is LPT scheduling */
    std::vector<double> cost(items.size());
    for (size_t i = 0; i < items.size(); ++i) {
        double c = 0;
        for (int s = items[i].seg_begin; s < items[i].seg_end; ++s) c += segs[s].type == dev::SEG_GEMM ? (double)segs[s].K : 1.0;
        cost[i] = c * items[i].tm * items[i].tn + 64.0;
    }
    std::vector<size_t> ord(items.size());
    for (size_t i = 0; i < ord.size(); ++i) ord[i] = i;
    const bool by_phase = item_phase.size() == items.size();
    std::stable_sort(ord.begin(), ord.end(), [&](size_t a, size_t b) {
        if (by_phase && item_phase[a] != item_phase[b]) return item_phase[a] < item_phase[b];
        return cost[a] > cost[b];
    });
    std::vector<dev::WorkItem> sorted(items.size());
    for (size_t i = 0; i < ord.size(); ++i) sorted[i] = items[ord[i]];
    items.swap(sorted);
    d_items = std::make_shared<DevBuf>(ctx, items.size() * sizeof(dev::WorkItem));
    d_segs = std::make_shared<DevBuf>(ctx, std::max<size_t>(1, segs.size()) * sizeof(dev::Segment));
    dev::h2d(ctx->st, d_items->p, items.data(), items.size() * sizeof(dev::WorkItem));
    dev::h2d(ctx->st, d_segs->p, segs.data(), segs.size() * sizeof(dev::Segment));
    if (!reduces.empty()) {
        d_reduces = std::make_shared<DevBuf>(ctx, reduces.size() * sizeof(dev::ReduceItem));
        dev::h2d(ctx->st, d_reduces->p, reduces.data(), reduces.size() * sizeof(dev::ReduceItem));
        scratch = std::make_shared<DevBuf>(ctx, (size_t)scratch_elems * 8);
    }
    dev::sync(ctx->st); /* the host vectors may be reallocated by the caller afterwards */
}

void Plan::run(Ctx* ctx, const double* x, double* y) const {
    if (items.empty()) return;
    double* w = scratch ? scratch->as<double>() : nullptr;
    dev::run_chain(ctx->st, d_items->as<dev::WorkItem>(), (int)items.size(), d_segs->as<dev::Segment>(), x, y, w);
    if (!reduces.empty()) dev::run_reduce(ctx->st, d_reduces->as<dev::ReduceItem>(), (int)reduces.size(), y, w);
}

static inline const double* padd(const double* p, long long elems) { return p + elems; }

void emit_cells(Plan& plan, double* C, bool c_in_y, long long ldc, int R, int Ncols, const std::vector<Contribution>& contribs,
                bool cover_all) {
    if (R <= 0 || Ncols <= 0) return;
    std::vector<int> rc = {0, R}, cc = {0, Ncols};
    for (const Contribution& c : contribs) {
        if (c.nr <= 0 || c.nc <= 0) continue;
        if (c.r0 < 0 || c.c0 < 0 || c.r0 + c.nr > R || c.c0 + c.nc > Ncols) throw Err(ERR_GENERIC, "emit_cells: contribution outside the panel");
        rc.push_back(c.r0); rc.push_back(c.r0 + c.nr);
        cc.push_back(c.c0); cc.push_back(c.c0 + c.nc);
    }
    std::sort(rc.begin(), rc.end()); rc.erase(std::unique(rc.begin(), rc.end()), rc.end());
    std::sort(cc.begin(), cc.end()); cc.erase(std::unique(cc.begin(), cc.end()), cc.end());
    for (size_t ri = 0; ri + 1 < rc.size(); ++ri) {
        const int r0 = rc[ri], r1 = rc[ri + 1];
        for (size_t ci = 0; ci + 1 < cc.size(); ++ci) {
            const int c0 = cc[ci], c1 = cc[ci + 1];
            const int seg_begin = (int)plan.segs.size();
            double kflops = 0;
            for (const Contribution& c : contribs) {
                if (c.nr <= 0 || c.nc <= 0) continue;
                if (!(c.r0 <= r0 && r1 <= c.r0 + c.nr && c.c0 <= c0 && c1 <= c.c0 + c.nc)) continue;
                dev::Segment s = c.seg;
                const long long dr = r0 - c.r0, dc = c0 - c.c0;
                switch (s.type) {
                    case dev::SEG_GEMM: s.A = padd(s.A, dr * s.lda_m); s.B = padd(s.B, dc * s.ldb_n); kflops += 2.0 * s.K; break;
                    case dev::SEG_AXPY: s.A = padd(s.A, dr * s.lda_m + dc * s.lda_k); break;
                    case dev::SEG_DIAG: s.d = (int)(s.d + dr - dc); break;
                    case dev::SEG_CSRA: s.row0 += (int)dr; s.A = padd(s.A, dc * s.ldb_n); break;
                    case dev::SEG_CSRB: s.row0 += (int)dc; s.A = padd(s.A, dr * s.lda_m); break;
                    case dev::SEG_CSRADD: s.row0 += (int)dr; s.d = (int)(s.d + dc); break;
                    default: throw Err(ERR_GENERIC, "emit_cells: bad segment type");
                }
                plan.segs.push_back(s);
            }
            const int seg_end = (int)plan.segs.size();
            if (seg_end == seg_begin && !cover_all) continue;
            const int M = r1 - r0, N = c1 - c0;
            /* tile extents in units of 16 rows/cols (two 8-row DMMA fragments, one per warp row), spread as evenly as
               possible over ceil(units/4) tiles: every tile is 64 or 48 (or less, for small cells) wide, and the two
               warp rows / columns of a CTA carry the same number of fragments */
            /* as many full 64-wide tiles as possible (they take the kernel's predicate-free path); the remainder is one
               ragged tile, merged with the last full tile and halved when that makes two tiles of at most 64 and at least
               40 (a sliver would waste a whole CTA on the fixed costs of a tile) */
            auto split = [](int len) {
                std::vector<int> ext;
                const int nfull = len / 64, rem = len % 64;
                for (int i = 0; i < nfull; ++i) ext.push_back(64);
                if (rem == 0) return ext;
                if (nfull > 0 && rem < 24) {
                    ext.pop_back();
                    const int tot = 64 + rem, h = (((tot + 1) / 2) + 7) / 8 * 8;
                    ext.push_back(h); ext.push_back(tot - h);
                } else ext.push_back(rem);
                return ext;
            };
            const std::vector<int> em = split(M), en = split(N);
            /* cut a long chain into parts of roughly equal K (whole segments only) */
            std::vector<int> part_begin = {seg_begin};
            if (plan.split_item_cost > 0 && seg_end - seg_begin > 1) {
                double ktot = 0;
                for (int sgi = seg_begin; sgi < seg_end; ++sgi) ktot += plan.segs[sgi].type == dev::SEG_GEMM ? plan.segs[sgi].K : 0;
                const double area = (double)em[0] * (double)en[0];
                int nparts = (int)std::ceil(ktot * area / plan.split_item_cost);
                nparts = std::max(1, std::min(nparts, seg_end - seg_begin));
                if (nparts > 1) {
                    double acc = 0;
                    int next = 1;
                    for (int sgi = seg_begin; sgi < seg_end && next < nparts; ++sgi) {
                        acc += plan.segs[sgi].type == dev::SEG_GEMM ? plan.segs[sgi].K : 0;
                        if (acc >= ktot * next / nparts && sgi + 1 < seg_end) { part_begin.push_back(sgi + 1); ++next; }
                    }
                }
            }
            part_begin.push_back(seg_end);
            const int nparts = (int)part_begin.size() - 1;
            int m0 = 0;
            for (int tm : em) {
                int n0 = 0;
                for (int tn : en) {
                    dev::WorkItem it;
                    std::memset(&it, 0, sizeof it);
                    it.m0 = m0; it.n0 = n0;
                    it.tm = tm; it.tn = tn;
                    it.mode = 0;
                    double* dst = C + (long long)(r0 + m0) * ldc + (c0 + n0);
                    {   /* FP64 tensor flops the kernel will EXECUTE for this tile: whole 8-row / 8-column fragments per warp half,
                           whole 16-deep K chunks (the useful count is plan.flops) */
                        auto frag = [](int t) { const int h = ((t + 15) >> 4) << 3; const int a = std::min(h, ((t + 7) / 8) * 8);
                                                const int b = std::max(0, std::min(h, ((t - h + 7) / 8) * 8)); return a + b; };
                        double kx = 0;
                        for (int sgi = seg_begin; sgi < seg_end; ++sgi)
                            if (plan.segs[sgi].type == dev::SEG_GEMM) kx += 16.0 * ((plan.segs[sgi].K + 15) / 16);
                        plan.exec_flops += 2.0 * frag(tm) * frag(tn) * kx;
                    }
                    if (nparts == 1) {
                        it.C = dst; it.ldc = ldc; it.c_in_y = c_in_y ? 1 : 0;
                        it.seg_begin = seg_begin; it.seg_end = seg_end;
                        plan.items.push_back(it);
                        plan.item_phase.push_back(0);
                    } else {
                        dev::ReduceItem ri;
                        std::memset(&ri, 0, sizeof ri);
                        ri.dst = dst; ri.ldc = ldc; ri.dst_in_y = c_in_y ? 1 : 0;
                        ri.src_off = plan.scratch_elems * 8; ri.tm = tm; ri.tn = tn; ri.nparts = nparts;
                        plan.reduces.push_back(ri);
                        for (int pp = 0; pp < nparts; ++pp) {
                            it.C = (double*)(uintptr_t)((plan.scratch_elems + (long long)pp * tm * tn) * 8);
                            it.ldc = tn; it.c_in_y = 2;
                            it.seg_begin = part_begin[pp]; it.seg_end = part_begin[pp + 1];
                            plan.items.push_back(it);
                            plan.item_phase.push_back(pp);
                        }
                        plan.scratch_elems += (long long)nparts * tm * tn;
                    }
                    n0 += tn;
                }
                m0 += tm;
            }
            plan.flops += kflops * (double)M * (double)N;
        }
    }
}

}  // namespace dmrgx
