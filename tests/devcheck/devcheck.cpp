/*  TEST-ONLY shim over csrc/dev.h for tests/test_device_kernels.py and tests/test_sparse_eig_kernels.py — NOT part of the product.
 *
 *  A thin extern "C" layer for ctypes: each entry point copies host arrays to the device, calls one dev:: function and
 *  copies the results back.  It is built twice (csrc/Makefile): libdevcheck_host.so links the host emulation of dev.h
 *  (tests/plancheck/dev_host*.cpp), libdevcheck_cuda.so links the product's own sm_100a object build/dev_cuda.o, so the
 *  same tests and tolerances run against both.
 *
 *  Guard bands.  Every host array handed in is [guard | payload | guard], with `guard` elements on each side; the whole
 *  array goes to the device and comes back, so the test sees what a kernel did to the guards.  The test fills operand
 *  guards and padding with NaN (an over-read shows up as NaN in a result) and output guards and gaps with a sentinel bit
 *  pattern (an over-write shows up as a changed sentinel).  The shim refuses a guard below 4 KiB or below one leading
 *  dimension of the buffer, so that reading one vector too many still lands inside the allocation.
 *
 *  Plan validation.  A chain plan arrives as records whose pointer fields are element offsets into one double pool and
 *  one int pool (CSR rowptr / colidx), or byte offsets into x / y / w where dev.h says so.  Before launching, the shim
 *  computes from the kernel's own addressing every element each (work item, segment) pair can touch — clamped rows
 *  included — and refuses a plan that reaches outside its buffer: a mistake in a test is an error return, never a fault.
 *
 *  Sparse-sector and eigensolver entries (dc_spmm, dc_syevd, tests/test_sparse_eig_kernels.py) follow the same rules; their
 *  conventions are stated above each of them.
 *
 *  Every entry point returns 0 or -1; dc_error() holds the message (a refusal of the shim, or what dev:: threw).
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "dev.h"

namespace {

using dev::Segment;
using dev::WorkItem;
using dev::ReduceItem;

static_assert(sizeof(Segment) == 96 && sizeof(WorkItem) == 48 && sizeof(ReduceItem) == 40, "record layouts of tests/test_device_kernels.py");
static_assert(sizeof(dev::SpTile) == 64 && sizeof(dev::SpASlot) == 64 && sizeof(dev::SpSSlot) == 64 && sizeof(dev::SpBSlot) == 112,
              "record layouts of tests/devcheck_common.py");

std::string g_msg;
dev::Stream* g_st = nullptr;

struct Refuse : std::runtime_error { using std::runtime_error::runtime_error; };
#define REFUSE_IF(cond, ...) do { if (cond) { char b_[400]; snprintf(b_, sizeof b_, __VA_ARGS__); throw Refuse(b_); } } while (0)

dev::Stream* stream() {
    if (!g_st && dev::init(0, nullptr, &g_st) != 0) { g_st = nullptr; throw std::runtime_error(std::string("dev::init: ") + dev::last_error()); }
    return g_st;
}

constexpr long long MIN_GUARD = 4096 / 8;

/* One host array [guard | payload | guard] mirrored on the device.  `need` payload elements must exist; `ld` is the
   leading dimension the guard must cover. */
template <class T>
struct Buf {
    T* host = nullptr;
    T* dev_base = nullptr;
    long long total = 0, guard = 0;
    bool out = false;
    Buf() = default;
    Buf(const Buf&) = delete;
    void set(T* h, long long tot, long long g, long long need, long long ld, bool is_out, const char* name) {
        if (!h) return;
        REFUSE_IF(g < MIN_GUARD || g < ld || (g & 1), "%s: guard of %lld elements is below 4 KiB, below the leading dimension %lld, or odd", name, g, ld);
        REFUSE_IF(need < 0 || tot < 2 * g + need, "%s: %lld elements hold no %lld-element payload between two %lld-element guards", name, tot, need, g);
        host = h; total = tot; guard = g; out = is_out;
        dev_base = (T*)dev::malloc_bytes(stream(), sizeof(T) * (size_t)tot);
        dev::h2d(stream(), dev_base, host, sizeof(T) * (size_t)tot);
    }
    long long n() const { return total - 2 * guard; }
    T* p() const { return dev_base ? dev_base + guard : nullptr; }
    void back() { if (dev_base && out) dev::d2h(stream(), host, dev_base, sizeof(T) * (size_t)total); }
    ~Buf() { if (dev_base) dev::free_bytes(g_st, dev_base); }
};

template <class F>
int guarded(F&& f) {
    try {
        f();
        return 0;
    } catch (const std::exception& e) {
        g_msg = e.what();
        return -1;
    }
}

/* --------------------------------------------------------------------------------------------------------------------
 *  chain plan validation: the element ranges of dev.h's addressing, per (work item, segment)
 * ------------------------------------------------------------------------------------------------------------------ */
struct Pools {
    long long nD, nI, nX, nY, nW, nO;
    const double* D; const int* I;
};

void in_range(long long lo, long long hi, long long n, const char* what, int item, int seg) {
    REFUSE_IF(lo < 0 || hi >= n, "item %d segment %d: %s reaches [%lld, %lld] outside its %lld-element buffer", item, seg, what, lo, hi, n);
}
/* an operand address field: element offset into D, or (flag set) byte offset into x */
void operand(long long field, bool in_x, long long lo, long long hi, const Pools& P, const char* what, int item, int seg) {
    if (in_x) {
        REFUSE_IF(field % 8, "item %d segment %d: %s byte offset %lld into x is not a multiple of 8", item, seg, what, field);
        in_range(field / 8 + lo, field / 8 + hi, P.nX, what, item, seg);
    } else in_range(field + lo, field + hi, P.nD, what, item, seg);
}

void check_chain(const WorkItem* items, int nitems, const Segment* segs, int nsegs, const ReduceItem* red, int nred, const Pools& P) {
    for (int w = 0; w < nitems; ++w) {
        const WorkItem& it = items[w];
        REFUSE_IF(it.tm < 1 || it.tn < 1 || it.tm > dev::TILE || it.tn > dev::TILE, "item %d: tile extents %dx%d", w, it.tm, it.tn);
        REFUSE_IF(it.seg_begin < 0 || it.seg_end < it.seg_begin || it.seg_end > nsegs, "item %d: segments [%d, %d) of %d", w, it.seg_begin, it.seg_end, nsegs);
        REFUSE_IF(it.mode < 0 || it.mode > 1 || it.c_in_y < 0 || it.c_in_y > 2 || it.ldc < it.tn || it.m0 < 0 || it.n0 < 0, "item %d: mode, c_in_y, ldc or origin", w);
        const long long c = (long long)(intptr_t)it.C, last = (long long)(it.tm - 1) * it.ldc + it.tn - 1;
        if (it.c_in_y == 0) in_range(c, c + last, P.nO, "C", w, -1);
        else {
            REFUSE_IF(c % 8, "item %d: C byte offset %lld is not a multiple of 8", w, c);
            in_range(c / 8, c / 8 + last, it.c_in_y == 1 ? P.nY : P.nW, it.c_in_y == 1 ? "C in y" : "C in w", w, -1);
        }
        for (int s = it.seg_begin; s < it.seg_end; ++s) {
            const Segment& sg = segs[s];
            const bool ax = sg.flags & dev::SEGF_A_X, bx = sg.flags & dev::SEGF_B_X;
            const long long A = (long long)(intptr_t)sg.A, B = (long long)(intptr_t)sg.B;
            REFUSE_IF(sg.lda_m < 0 || sg.lda_k < 0 || sg.ldb_n < 0 || sg.ldb_k < 0 || sg.K < 0, "item %d segment %d: negative stride or K", w, s);
            const long long m0 = it.m0, m1 = it.m0 + it.tm - 1, n0 = it.n0, n1 = it.n0 + it.tn - 1;
            auto csr_rows = [&](long long r0, long long r1, auto&& per_entry) {
                const long long rp = (long long)(intptr_t)sg.rowptr, ci = (long long)(intptr_t)sg.colidx;
                in_range(rp + r0, rp + r1 + 1, P.nI, "rowptr", w, s);
                for (long long r = r0; r <= r1; ++r) {
                    const int e0 = P.I[rp + r], e1 = P.I[rp + r + 1];
                    if (e1 <= e0) continue;
                    in_range(ci + e0, ci + e1 - 1, P.nI, "colidx", w, s);
                    operand(B, bx, e0, e1 - 1, P, "CSR values", w, s);
                    for (int e = e0; e < e1; ++e) per_entry((long long)P.I[ci + e]);
                }
            };
            switch (sg.type) {
                case dev::SEG_GEMM:
                    if (sg.K == 0) break;
                    operand(A, ax, m0 * sg.lda_m, m1 * sg.lda_m + (sg.K - 1) * sg.lda_k, P, "A", w, s);
                    operand(B, bx, n0 * sg.ldb_n, n1 * sg.ldb_n + (sg.K - 1) * sg.ldb_k, P, "B", w, s);
                    break;
                case dev::SEG_AXPY: operand(A, ax, m0 * sg.lda_m + n0 * sg.lda_k, m1 * sg.lda_m + n1 * sg.lda_k, P, "A", w, s); break;
                case dev::SEG_DIAG: break;
                case dev::SEG_CSRA:
                    csr_rows(sg.row0 + m0, sg.row0 + m1, [&](long long col) {
                        REFUSE_IF(col < 0, "item %d segment %d: negative column", w, s);
                        operand(A, ax, col * sg.ldb_k + n0 * sg.ldb_n, col * sg.ldb_k + n1 * sg.ldb_n, P, "CSRA dense factor", w, s);
                    });
                    break;
                case dev::SEG_CSRB:
                    csr_rows(sg.row0 + n0, sg.row0 + n1, [&](long long col) {
                        REFUSE_IF(col < 0, "item %d segment %d: negative column", w, s);
                        operand(A, ax, m0 * sg.lda_m + col * sg.lda_k, m1 * sg.lda_m + col * sg.lda_k, P, "CSRB dense factor", w, s);
                    });
                    break;
                case dev::SEG_CSRADD: csr_rows(sg.row0 + m0, sg.row0 + m1, [](long long) {}); break;
                default: REFUSE_IF(true, "item %d segment %d: type %d", w, s, sg.type);
            }
        }
    }
    for (int r = 0; r < nred; ++r) {
        const ReduceItem& it = red[r];
        REFUSE_IF(it.tm < 1 || it.tn < 1 || it.nparts < 1 || it.ldc < it.tn || it.src_off % 8, "reduce item %d: extents, parts, ldc or source offset", r);
        const long long d = (long long)(intptr_t)it.dst, last = (long long)(it.tm - 1) * it.ldc + it.tn - 1;
        if (it.dst_in_y) { REFUSE_IF(d % 8, "reduce item %d: byte offset", r); in_range(d / 8, d / 8 + last, P.nY, "reduce dst in y", r, -1); }
        else in_range(d, d + last, P.nO, "reduce dst", r, -1);
        in_range(it.src_off / 8, it.src_off / 8 + (long long)it.nparts * it.tm * it.tn - 1, P.nW, "reduce parts in w", r, -1);
    }
}

}  // namespace

extern "C" {

const char* dc_error() { return g_msg.c_str(); }
long long dc_min_guard() { return MIN_GUARD; }

/* One run_chain launch (then run_reduce when nred > 0) on pools D (doubles), I (ints), X, Y, W and O (plain outputs).
   Pointer fields: see the header comment; Y, W and O come back. */
int dc_chain(const void* items, int nitems, const void* segs, int nsegs, const void* red, int nred, long long guard, double* D, long long nD, int* I,
             long long nI, double* X, long long nX, double* Y, long long nY, double* W, long long nW, double* O, long long nO) {
    return guarded([&] {
        REFUSE_IF(nitems < 1 && nred < 1, "nothing to run");
        Buf<double> d, x, y, w, o;
        Buf<int> ib;
        d.set(D, nD, guard, 0, 0, false, "D"); ib.set(I, nI, guard, 0, 0, false, "I");
        x.set(X, nX, guard, 0, 0, false, "X"); y.set(Y, nY, guard, 0, 0, true, "Y");
        w.set(W, nW, guard, 0, 0, true, "W"); o.set(O, nO, guard, 0, 0, true, "O");
        const Pools P{d.n(), ib.n(), x.n(), y.n(), w.n(), o.n(), D + guard, I + guard};
        std::vector<WorkItem> it((const WorkItem*)items, (const WorkItem*)items + nitems);
        std::vector<Segment> sg((const Segment*)segs, (const Segment*)segs + nsegs);
        std::vector<ReduceItem> rd((const ReduceItem*)red, (const ReduceItem*)red + nred);
        check_chain(it.data(), nitems, sg.data(), nsegs, rd.data(), nred, P);
        /* rebase: element offsets into D / I become device pointers; byte offsets into x / y / w stay as they are */
        for (auto& s : sg) {
            if (!(s.flags & dev::SEGF_A_X)) s.A = d.p() + (intptr_t)s.A;
            if (!(s.flags & dev::SEGF_B_X)) s.B = d.p() + (intptr_t)s.B;
            s.rowptr = ib.p() + (intptr_t)s.rowptr;
            s.colidx = ib.p() + (intptr_t)s.colidx;
        }
        for (auto& t : it) if (t.c_in_y == 0) t.C = o.p() + (intptr_t)t.C;
        for (auto& r : rd) if (!r.dst_in_y) r.dst = o.p() + (intptr_t)r.dst;
        dev::Stream* st = stream();
        Buf<WorkItem> di; Buf<Segment> ds; Buf<ReduceItem> dr;
        auto upload = [&](auto& b, auto& v) {
            using T = typename std::decay_t<decltype(v)>::value_type;
            if (v.empty()) return;
            b.dev_base = (T*)dev::malloc_bytes(st, sizeof(T) * v.size());
            dev::h2d(st, b.dev_base, v.data(), sizeof(T) * v.size());
        };
        upload(di, it); upload(ds, sg); upload(dr, rd);
        if (nitems > 0) dev::run_chain(st, di.dev_base, nitems, ds.dev_base, x.p(), y.p(), w.p());
        if (nred > 0) dev::run_reduce(st, dr.dev_base, nred, y.p(), w.p());
        y.back(); w.back(); o.back();
        dev::sync(st);
    });
}

/* G = PᵀP: P holds np columns of ldp doubles; `shift` moves the column base by that many doubles (alignment checks) */
int dc_gram(double* P, long long nP, long long ldp, int np, long long n, int shift, double* G, long long nG, long long guard) {
    return guarded([&] {
        REFUSE_IF(np < 1 || n < 0 || ldp < n || shift < 0 || shift > 1, "np, n, ldp or shift");
        Buf<double> p, g;
        p.set(P, nP, guard, (np - 1) * ldp + n + shift, ldp, false, "P");
        g.set(G, nG, guard, (long long)np * np, np, true, "G");
        dev::gram(stream(), p.p() + shift, ldp, np, n, g.p());
        g.back();
        dev::sync(stream());
    });
}

/* gs_pass; coef, dots and nrm2 may each be null.  w and the outputs come back. */
int dc_gs_pass(double* V, long long nV, long long ldv, int nvec, double* w, long long nw, long long n, double* coef, long long ncoef, double* dots,
               long long ndots, double* nrm2, long long nnrm2, long long guard) {
    return guarded([&] {
        REFUSE_IF(nvec < 1 || n < 0 || ldv < n, "nvec, n or ldv");
        Buf<double> v, x, c, d, r;
        v.set(V, nV, guard, (nvec - 1) * ldv + n, ldv, false, "V");
        x.set(w, nw, guard, n, 0, true, "w");
        c.set(coef, ncoef, guard, nvec, 0, false, "coef");
        d.set(dots, ndots, guard, nvec, 0, true, "dots");
        r.set(nrm2, nnrm2, guard, 1, 0, true, "nrm2");
        dev::gs_pass(stream(), v.p(), ldv, nvec, x.p(), n, c.p(), d.p(), r.p());
        x.back(); d.back(); r.back();
        dev::sync(stream());
    });
}

int dc_gs_final(double* V, long long nV, long long ldv, int nvec, double* w, long long nw, long long n, double* coef, long long ncoef, double* nrm2_in,
                long long nin, double* nrm2_out, long long nout, double* vout, long long nvout, long long guard) {
    return guarded([&] {
        REFUSE_IF(nvec < 1 || n < 0 || ldv < n, "nvec, n or ldv");
        Buf<double> v, x, c, ri, ro, o;
        v.set(V, nV, guard, (nvec - 1) * ldv + n, ldv, false, "V");
        x.set(w, nw, guard, n, 0, false, "w");
        c.set(coef, ncoef, guard, nvec, 0, false, "coef");
        ri.set(nrm2_in, nin, guard, 1, 0, false, "nrm2_in");
        ro.set(nrm2_out, nout, guard, 1, 0, true, "nrm2_out");
        o.set(vout, nvout, guard, n, 0, true, "vout");
        dev::gs_final(stream(), v.p(), ldv, nvec, x.p(), n, c.p(), ri.p(), ro.p(), o.p());
        ro.back(); o.back();
        dev::sync(stream());
    });
}

int dc_dot(double* x, long long nx, double* y, long long ny, long long n, double* out, long long nout, long long guard) {
    return guarded([&] {
        Buf<double> a, b, o;
        a.set(x, nx, guard, n, 0, false, "x");
        b.set(y, ny, guard, n, 0, false, "y");
        o.set(out, nout, guard, 1, 0, true, "out");
        dev::dot(stream(), a.p(), b.p(), n, o.p());
        o.back();
        dev::sync(stream());
    });
}

int dc_scale_inv_norm(double* w, long long nw, double* nrm2, long long nn, double* v, long long nv, long long n, long long guard) {
    return guarded([&] {
        Buf<double> a, r, o;
        a.set(w, nw, guard, n, 0, false, "w");
        r.set(nrm2, nn, guard, 1, 0, false, "nrm2");
        o.set(v, nv, guard, n, 0, true, "v");
        dev::scale_inv_norm(stream(), a.p(), r.p(), o.p(), n);
        o.back();
        dev::sync(stream());
    });
}

int dc_ritz_rotate(double* V, long long nV, long long ldv, long long n, int ncv, double* S, long long nS, int kk, long long guard) {
    return guarded([&] {
        REFUSE_IF(ncv < 1 || kk < 1 || kk > ncv || n < 0 || ldv < n, "ncv, kk, n or ldv");
        Buf<double> v, s;
        v.set(V, nV, guard, (ncv - 1) * ldv + n, ldv, true, "V");
        s.set(S, nS, guard, (long long)ncv * kk, 0, false, "S");
        dev::ritz_rotate(stream(), v.p(), ldv, n, ncv, s.p(), kk);
        v.back();
        dev::sync(stream());
    });
}

int dc_lanczos_blocks(long long n) { return dev::lanczos_blocks(n); }

/* One lanczos_batch pass.  Per-column state (nb, or nb × nsteps for alpha / beta) in and out; the block partials are a
   NaN-filled scratch of the shim, so a sum that read a partial before it was written turns NaN. */
int dc_lanczos(int pass, int t, int nb, int nsteps, long long n, long long ld, double* alpha, double* beta, double* norm2, long long* ndone,
               double* a, double* scale, double* zero2, int* done, unsigned* tickets, long long nstate, double* prev, double* cur, double* y,
               long long nvec, long long guard) {
    return guarded([&] {
        REFUSE_IF(nb < 1 || nsteps < 1 || n < 1 || pass < 0 || pass > 2 || t < 0 || t >= nsteps, "nb, nsteps, n, pass or t");
        const long long cols = (nb - 1) * ld + n, ns = (long long)nb * nsteps;
        Buf<double> al, be, nm, aa, sc, z, pv, cu, yy;
        Buf<long long> nd;
        Buf<int> dn;
        Buf<unsigned> tk;
        al.set(alpha, ns + 2 * guard, guard, ns, 0, true, "alpha");
        be.set(beta, ns + 2 * guard, guard, ns, 0, true, "beta");
        nm.set(norm2, nstate, guard, nb, 0, true, "norm2");
        nd.set(ndone, nstate, guard, nb, 0, true, "ndone");
        aa.set(a, nstate, guard, nb, 0, true, "a");
        sc.set(scale, nstate, guard, nb, 0, true, "scale");
        z.set(zero2, nstate, guard, nb, 0, false, "zero2");
        dn.set(done, nstate, guard, nb, 0, true, "done");
        tk.set(tickets, nstate, guard, nb, 0, true, "tickets");
        pv.set(prev, nvec, guard, cols, ld, false, "prev");
        cu.set(cur, nvec, guard, cols, ld, true, "cur");
        yy.set(y, nvec, guard, cols, ld, true, "y");
        const long long np = (long long)nb * dev::lanczos_blocks(n);
        std::vector<double> nan((size_t)np, std::nan(""));
        Buf<double> part;
        part.dev_base = (double*)dev::malloc_bytes(stream(), sizeof(double) * (size_t)np);
        dev::h2d(stream(), part.dev_base, nan.data(), sizeof(double) * (size_t)np);
        dev::LanczosBatch L;
        L.nb = nb; L.nsteps = nsteps; L.n = n; L.ld = ld;
        L.alpha = al.p(); L.beta = be.p(); L.norm2 = nm.p(); L.ndone = nd.p(); L.a = aa.p(); L.scale = sc.p(); L.zero2 = z.p(); L.done = dn.p();
        L.partials = part.dev_base; L.tickets = tk.p();
        dev::lanczos_batch(stream(), L, pass, t, pv.p(), cu.p(), yy.p());
        al.back(); be.back(); nm.back(); nd.back(); aa.back(); sc.back(); dn.back(); tk.back(); cu.back(); yy.back();
        dev::sync(stream());
    });
}

int dc_fill_random(double* x, long long nx, long long n, unsigned long long seed, long long first, long long guard) {
    return guarded([&] {
        Buf<double> o;
        o.set(x, nx, guard, n, 0, true, "x");
        dev::fill_random(stream(), o.p(), n, seed, first);
        o.back();
        dev::sync(stream());
    });
}

int dc_filter_small(double* x, long long nx, long long n, double tol, long long guard) {
    return guarded([&] {
        Buf<double> o;
        o.set(x, nx, guard, n, 0, true, "x");
        dev::filter_small(stream(), o.p(), n, tol);
        o.back();
        dev::sync(stream());
    });
}

int dc_axpby_out(double* a, long long na, double* b, long long nb, double alpha, double* out, long long nout, long long n, long long guard) {
    return guarded([&] {
        Buf<double> x, y, o;
        x.set(a, na, guard, n, 0, false, "a");
        y.set(b, nb, guard, n, 0, false, "b");
        o.set(out, nout, guard, n, 0, true, "out");
        dev::axpby_out(stream(), x.p(), y.p(), alpha, o.p(), n);
        o.back();
        dev::sync(stream());
    });
}

int dc_gather_rows_reversed(double* src, long long nsrc, int n, int m, double* dst, long long ndst, long long guard) {
    return guarded([&] {
        REFUSE_IF(n < 1 || m < 0 || m > n, "n or m");
        Buf<double> s, d;
        s.set(src, nsrc, guard, (long long)n * n, n, false, "src");
        d.set(dst, ndst, guard, (long long)m * n, n, true, "dst");
        dev::gather_rows_reversed(stream(), s.p(), n, m, d.p());
        d.back();
        dev::sync(stream());
    });
}

/* One run_spmm launch over the pools X (psi, read), Y (written at X's offsets), I (ELL columns) and V (ELL values).
   Offsets as in the product: SpTile.off, SpASlot.src and SpBSlot.src are element offsets into X (and Y); SpBSlot.ecol
   and .eval arrive as element offsets into I and V and are rebased here.  Validation covers every address spmm_kernel
   forms, including the rows r >= nrows of a partial tile that it reads (but never writes) and the shared-memory stage
   of SP_ROWS·max_nR doubles that its in-tile offsets index.  Y comes back. */
int dc_spmm(const void* tiles, int ntiles, const void* aslots, int na, const void* sslots, int ns, const void* bslots, int nb, long long guard, double* X,
            long long nX, double* Y, long long nY, int* I, long long nI, double* V, long long nV, int max_nR) {
    return guarded([&] {
        using dev::SP_ROWS;
        REFUSE_IF(ntiles < 0 || na < 0 || ns < 0 || nb < 0 || max_nR < 1, "ntiles, slot counts or max_nR");
        REFUSE_IF(guard < (long long)SP_ROWS * max_nR, "Y: guard of %lld elements is below SP_ROWS·max_nR = %lld", guard, (long long)SP_ROWS * max_nR);
        Buf<double> x, y, v;
        Buf<int> ib;
        x.set(X, nX, guard, 1, 0, false, "X"); y.set(Y, nY, guard, 1, 0, true, "Y");
        ib.set(I, nI, guard, 1, 0, false, "I"); v.set(V, nV, guard, 1, 0, false, "V");
        const long long px = x.n(), stage = (long long)SP_ROWS * max_nR;
        const int* Ih = I + guard;
        std::vector<dev::SpTile> tl((const dev::SpTile*)tiles, (const dev::SpTile*)tiles + ntiles);
        std::vector<dev::SpASlot> as((const dev::SpASlot*)aslots, (const dev::SpASlot*)aslots + na);
        std::vector<dev::SpSSlot> ss((const dev::SpSSlot*)sslots, (const dev::SpSSlot*)sslots + ns);
        std::vector<dev::SpBSlot> bs((const dev::SpBSlot*)bslots, (const dev::SpBSlot*)bslots + nb);
        auto in_x = [&](long long lo, long long n, int w, const char* what) {
            REFUSE_IF(lo < 0 || lo + n > px, "tile %d: %s [%lld, %lld) outside the %lld-element X", w, what, lo, lo + n, px);
        };
        /* an in-tile offset: inside the staged rows for r < nrows, inside the shared-memory stage for r >= nrows */
        auto in_tile = [&](long long lo, long long hi, int r, const dev::SpTile& t, int w, const char* what) {
            const long long lim = r < t.nrows ? (long long)t.nrows * t.nR : stage;
            REFUSE_IF(lo < 0 || hi >= lim, "tile %d row %d: %s [%lld, %lld] outside [0, %lld)", w, r, what, lo, hi, lim);
        };
        for (int w = 0; w < ntiles; ++w) {
            const dev::SpTile& t = tl[(size_t)w];
            REFUSE_IF(t.nrows < 1 || t.nrows > SP_ROWS || t.nR < 1 || t.nR > max_nR, "tile %d: nrows %d or nR %d (max_nR %d)", w, t.nrows, t.nR, max_nR);
            in_x(t.off, (long long)t.nrows * t.nR, w, "rows");
            REFUSE_IF(t.off + (long long)t.nrows * t.nR > y.n(), "tile %d: rows outside Y", w);
            REFUSE_IF(t.a_begin < 0 || t.a_count < 0 || t.a_begin + t.a_count > na || t.s_begin < 0 || t.s_count < 0 || t.s_begin + t.s_count > ns ||
                          t.b_begin < 0 || t.b_count < 0 || t.b_begin + t.b_count > nb, "tile %d: slot ranges", w);
            for (int k = t.a_begin; k < t.a_begin + t.a_count; ++k)
                for (int r = 0; r < SP_ROWS; ++r) in_x(as[(size_t)k].src[r], t.nR, w, "a-slot source row");
            for (int k = t.s_begin; k < t.s_begin + t.s_count; ++k)
                for (int r = 0; r < SP_ROWS; ++r) in_tile(ss[(size_t)k].roff[r], ss[(size_t)k].roff[r] + t.nR - 1LL, r, t, w, "s-slot source row");
            for (int k = t.b_begin; k < t.b_begin + t.b_count; ++k) {
                const dev::SpBSlot& b = bs[(size_t)k];
                REFUSE_IF(b.W < 0 || b.ld < t.nR, "tile %d b-slot %d: W %d or ld %d below nR %d", w, k, b.W, b.ld, t.nR);
                if (b.W == 0) continue;
                const long long e0 = (long long)(intptr_t)b.ecol, v0 = (long long)(intptr_t)b.eval, span = (long long)(b.W - 1) * b.ld + t.nR;
                REFUSE_IF(e0 < 0 || e0 + span > ib.n() || v0 < 0 || v0 + span > v.n(), "tile %d b-slot %d: ELL columns or values outside I / V", w, k);
                int cmin = 0x7fffffff, cmax = -1;
                for (int q = 0; q < b.W; ++q)
                    for (int c = 0; c < t.nR; ++c) { const int col = Ih[e0 + (long long)q * b.ld + c]; cmin = std::min(cmin, col); cmax = std::max(cmax, col); }
                REFUSE_IF(cmin < 0, "tile %d b-slot %d: negative column", w, k);
                for (int r = 0; r < SP_ROWS; ++r) {
                    if (b.all_in) in_tile((long long)b.roff[r] + cmin, (long long)b.roff[r] + cmax, r, t, w, "all_in gather");
                    else in_x(b.src[r] + cmin, cmax - cmin + 1LL, w, "b-slot gather");
                }
            }
        }
        for (auto& b : bs) { b.ecol = ib.p() + (intptr_t)b.ecol; b.eval = v.p() + (intptr_t)b.eval; }
        dev::Stream* st = stream();
        Buf<dev::SpTile> dt; Buf<dev::SpASlot> da; Buf<dev::SpSSlot> ds; Buf<dev::SpBSlot> db;
        auto upload = [&](auto& buf, auto& vec) {   /* at least one record, as the product allocates */
            using T = typename std::decay_t<decltype(vec)>::value_type;
            buf.dev_base = (T*)dev::malloc_bytes(st, sizeof(T) * std::max<size_t>(1, vec.size()));
            dev::h2d(st, buf.dev_base, vec.data(), sizeof(T) * vec.size());
        };
        upload(dt, tl); upload(da, as); upload(ds, ss); upload(db, bs);
        dev::run_spmm(st, dt.dev_base, ntiles, da.dev_base, ds.dev_base, db.dev_base, x.p(), y.p(), max_nR);
        y.back();
        dev::sync(st);
    });
}

/* One syevd_batch call on nblocks blocks: block b is n[b]×n[b] at element offset a_off[b] of the pool A, its eigenvalues
   go to w_off[b] of W.  The pools are uploaded and read back whole with the shim's async copies on the main stream and no
   synchronisation before the call, so the solver runs ordered after queued work as dev.h promises.  A payload closer than
   `guard` elements to another payload or to an end of its pool is refused. */
int dc_syevd(int nblocks, const int* n, const long long* a_off, const long long* w_off, double* A, long long nA, double* W, long long nW, long long guard) {
    return guarded([&] {
        REFUSE_IF(nblocks < 0 || guard < MIN_GUARD, "nblocks, or guard below 4 KiB");
        auto check_pool = [&](const long long* off, bool square, long long total, const char* name) {
            std::vector<std::pair<long long, long long>> iv;
            for (int b = 0; b < nblocks; ++b) {
                REFUSE_IF(n[b] < 0, "block %d: n %d", b, n[b]);
                iv.push_back({off[b], off[b] + (square ? (long long)n[b] * n[b] : n[b])});
            }
            std::sort(iv.begin(), iv.end());
            long long end = 0;   /* the pool's start counts as a payload ending at 0 */
            for (auto& p : iv) {
                REFUSE_IF(p.first < end + guard, "%s: a payload at %lld is closer than %lld elements to the previous payload or the pool start", name, p.first, guard);
                end = std::max(end, p.second);
            }
            REFUSE_IF(end + guard > total, "%s: a payload ends closer than %lld elements to the pool end (%lld elements)", name, guard, total);
        };
        check_pool(a_off, true, nA, "A");
        check_pool(w_off, false, nW, "W");
        dev::Stream* st = stream();
        double* dA = (double*)dev::malloc_bytes(st, sizeof(double) * (size_t)nA);
        double* dW = (double*)dev::malloc_bytes(st, sizeof(double) * (size_t)nW);
        struct Free { double *a, *w; ~Free() { dev::free_bytes(g_st, a); dev::free_bytes(g_st, w); } } fr{dA, dW};
        dev::h2d(st, dA, A, sizeof(double) * (size_t)nA);
        dev::h2d(st, dW, W, sizeof(double) * (size_t)nW);
        std::vector<double*> pa((size_t)nblocks), pw((size_t)nblocks);
        for (int b = 0; b < nblocks; ++b) { pa[(size_t)b] = dA + a_off[b]; pw[(size_t)b] = dW + w_off[b]; }
        const int rc = dev::syevd_batch(st, nblocks, n, pa.data(), pw.data());
        dev::d2h(st, A, dA, sizeof(double) * (size_t)nA);
        dev::d2h(st, W, dW, sizeof(double) * (size_t)nW);
        dev::sync(st);
        REFUSE_IF(rc != 0, "syevd_batch returned %d: %s", rc, dev::last_error());
    });
}

}  // extern "C"
