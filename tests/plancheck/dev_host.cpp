/*  TEST-ONLY host emulation of csrc/dev.h — NOT part of the product.
 *
 *  libdmrgx_b200.so links dev_cuda.cu and fails loudly without a CUDA device.  This file exists so that
 *  `pytest -m "not gpu"` can exercise the HOST planning logic of the product (tile classification,
 *  sector/offset maps, work-item and segment lists, Lanczos restart logic, truncation selection) in a
 *  container without a GPU: it interprets the very same work lists with naive scalar loops over host
 *  memory.  It is built into tests/plancheck/libdmrgx_plancheck.so by tests/plancheck/Makefile and is
 *  loaded only by tests that say so; bench.py, smoke() and the C-ABI product library never see it.
 */
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "dev.h"

namespace dev {

struct Stream { int device; };
static std::string g_err;
static long long g_launches = 0;
const char* last_error() { return g_err.c_str(); }
long long launch_count() { return g_launches; }
int init(int device, void*, Stream** out) { *out = new Stream{device}; return 0; }
void destroy(Stream* s) { delete s; }
void make_current(Stream*) {}
void* malloc_bytes(Stream*, size_t b) { return std::malloc(b ? b : 8); }
void free_bytes(Stream*, void* p) { std::free(p); }
void h2d(Stream*, void* d, const void* s, size_t b) { if (b) std::memcpy(d, s, b); }
void d2h(Stream*, void* d, const void* s, size_t b) { if (b) std::memcpy(d, s, b); }
void d2d(Stream*, void* d, const void* s, size_t b) { if (b) std::memmove(d, s, b); }
void memset0(Stream*, void* d, size_t b) { if (b) std::memset(d, 0, b); }
void sync(Stream*) {}

/* Preconditions of the sm_100a kernels, checked here so that a host plan the GPU would refuse or mishandle fails on the
   CPU too.  chain_kernel's Stager keeps the element offsets of a thread's staged elements in 32-bit ints: within one
   16-deep chunk the farthest is (extent - 1)·ld_row + (min(K, 16) - 1)·ld_k, for A (rows, lda_m, lda_k) and B (columns,
   ldb_n, ldb_k) of every GEMM segment. */
static void check_stager(long long ext, long long ld_row, long long ld_k, int K, int item, int seg, const char* op) {
    const long long far = (ext - 1) * ld_row + (long long)(std::min(K, 16) - 1) * ld_k;
    if (ld_row < 0 || ld_k < 0 || far > 2147483647LL)
        throw std::runtime_error("run_chain: item " + std::to_string(item) + " segment " + std::to_string(seg) + ": the " + op +
                                 " staging offset " + std::to_string(far) + " does not fit the kernel's 32-bit Stager offsets");
}
void check_chain_plan(const WorkItem* items, int nitems, const Segment* segs) {
    for (int w = 0; w < nitems; ++w) {
        const WorkItem& it = items[w];
        if (it.tm < 1 || it.tn < 1 || it.tm > TILE || it.tn > TILE) throw std::runtime_error("run_chain: bad tile extents");
        for (int s = it.seg_begin; s < it.seg_end; ++s) {
            const Segment& sg = segs[s];
            if (sg.type != SEG_GEMM || sg.K <= 0) continue;
            check_stager(it.tm, sg.lda_m, sg.lda_k, sg.K, w, s, "A");
            check_stager(it.tn, sg.ldb_n, sg.ldb_k, sg.K, w, s, "B");
        }
    }
}

void run_chain(Stream*, const WorkItem* items, int nitems, const Segment* segs, const double* xbase, double* ybase, double* wbase) {
    ++g_launches;
    check_chain_plan(items, nitems, segs);
    std::vector<double> acc;
    for (int w = 0; w < nitems; ++w) {
        WorkItem it = items[w];
        if (it.c_in_y) it.C = (double*)((char*)(it.c_in_y == 1 ? ybase : wbase) + (size_t)it.C);
        acc.assign((size_t)it.tm * it.tn, 0.0);
        for (int s = it.seg_begin; s < it.seg_end; ++s) {
            Segment sg = segs[s];
            if (sg.flags & SEGF_A_X) sg.A = (const double*)((const char*)xbase + (size_t)sg.A);
            if (sg.flags & SEGF_B_X) sg.B = (const double*)((const char*)xbase + (size_t)sg.B);
            for (int m = 0; m < it.tm; ++m)
                for (int n = 0; n < it.tn; ++n) {
                    const long long gm = it.m0 + m, gn = it.n0 + n;
                    double v = 0.0;
                    switch (sg.type) {
                        case SEG_GEMM:
                            for (int k = 0; k < sg.K; ++k) v += sg.A[gm * sg.lda_m + k * sg.lda_k] * sg.B[gn * sg.ldb_n + k * sg.ldb_k];
                            break;
                        case SEG_AXPY: v = sg.A[gm * sg.lda_m + gn * sg.lda_k]; break;
                        case SEG_DIAG: v = (gm + sg.d == gn) ? 1.0 : 0.0; break;
                        case SEG_CSRA: {
                            const int r = sg.row0 + (int)gm;
                            for (int e = sg.rowptr[r]; e < sg.rowptr[r + 1]; ++e) v += sg.B[e] * sg.A[(long long)sg.colidx[e] * sg.ldb_k + gn * sg.ldb_n];
                        } break;
                        case SEG_CSRB: {
                            const int r = sg.row0 + (int)gn;
                            for (int e = sg.rowptr[r]; e < sg.rowptr[r + 1]; ++e) v += sg.B[e] * sg.A[gm * sg.lda_m + (long long)sg.colidx[e] * sg.lda_k];
                        } break;
                        case SEG_CSRADD: {
                            const int r = sg.row0 + (int)gm;
                            for (int e = sg.rowptr[r]; e < sg.rowptr[r + 1]; ++e) if (sg.colidx[e] == (int)gn + sg.d) v += sg.B[e];
                        } break;
                        default: throw std::runtime_error("bad segment type");
                    }
                    acc[(size_t)m * it.tn + n] += sg.coef * v;
                }
        }
        for (int m = 0; m < it.tm; ++m)
            for (int n = 0; n < it.tn; ++n) {
                double* p = it.C + (long long)m * it.ldc + n;
                if (it.mode == 0) *p = acc[(size_t)m * it.tn + n]; else *p += acc[(size_t)m * it.tn + n];
            }
    }
}

void run_spmm(Stream*, const SpTile* tiles, int ntiles, const SpASlot* aslots, const SpSSlot* sslots, const SpBSlot* bslots, const double* x, double* y, int max_nR) {
    ++g_launches;
    if (ntiles <= 0) return;
    /* the kernel stages a tile's rows in SP_ROWS·max_nR doubles of shared memory */
    if (max_nR > SP_MAX_NR) throw std::runtime_error("run_spmm: max_nR " + std::to_string(max_nR) + " exceeds SP_MAX_NR");
    for (int w = 0; w < ntiles; ++w)
        if (tiles[w].nR > max_nR || tiles[w].nrows > SP_ROWS) throw std::runtime_error("run_spmm: tile " + std::to_string(w) + " is wider than max_nR or taller than SP_ROWS");
    for (int w = 0; w < ntiles; ++w) {
        const SpTile& tl = tiles[w];
        for (int r = 0; r < tl.nrows; ++r)
            for (int c = 0; c < tl.nR; ++c) {
                double acc = 0.0;
                for (int k = 0; k < tl.a_count; ++k) { const SpASlot& S = aslots[tl.a_begin + k]; acc += S.w[r] * x[S.src[r] + c]; }
                for (int k = 0; k < tl.s_count; ++k) { const SpSSlot& S = sslots[tl.s_begin + k]; acc += S.w[r] * x[tl.off + S.roff[r] + c]; }
                for (int k = 0; k < tl.b_count; ++k) {
                    const SpBSlot& S = bslots[tl.b_begin + k];
                    double a = 0.0;
                    const long long base = S.all_in ? tl.off + S.roff[r] : S.src[r];
                    for (int t = 0; t < S.W; ++t) a += S.eval[(long long)t * S.ld + c] * x[base + S.ecol[(long long)t * S.ld + c]];
                    acc += S.w[r] * a;
                }
                y[tl.off + (long long)r * tl.nR + c] = acc;
            }
    }
}

void run_reduce(Stream*, const ReduceItem* items, int nitems, double* ybase, const double* wbase) {
    ++g_launches;
    for (int i = 0; i < nitems; ++i) {
        const ReduceItem& it = items[i];
        double* dst = it.dst_in_y ? (double*)((char*)ybase + (size_t)it.dst) : it.dst;
        const double* src = (const double*)((const char*)wbase + it.src_off);
        const int cnt = it.tm * it.tn;
        for (int e = 0; e < cnt; ++e) {
            double v = src[e];
            for (int p = 1; p < it.nparts; ++p) v += src[(long long)p * cnt + e];
            dst[(long long)(e / it.tn) * it.ldc + (e % it.tn)] = v;
        }
    }
}

static unsigned long long splitmix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
void fill_random(Stream*, double* x, long long n, unsigned long long seed, long long first) {
    ++g_launches;
    for (long long i = 0; i < n; ++i) x[i] = (double)(splitmix64(seed + (unsigned long long)(first + i) * 0x9E3779B97F4A7C15ULL) >> 11) / 9007199254740992.0 - 0.5;
}
void dot(Stream*, const double* x, const double* y, long long n, double* out) {
    ++g_launches;
    double s = 0;
    for (long long q = 0; q < n; ++q) s += x[q] * y[q];
    *out = s;
}
void gs_pass(Stream*, const double* V, long long ldv, int nvec, double* w, long long n, const double* coef, double* dots, double* nrm2) {
    ++g_launches;
    if (nvec > MAX_BASIS) throw std::runtime_error("gs_pass: nvec " + std::to_string(nvec) + " exceeds MAX_BASIS");
    if (coef) for (int i = 0; i < nvec; ++i) for (long long q = 0; q < n; ++q) w[q] -= coef[i] * V[i * ldv + q];
    if (dots) for (int i = 0; i < nvec; ++i) { double s = 0; for (long long q = 0; q < n; ++q) s += V[i * ldv + q] * w[q]; dots[i] = s; }
    if (nrm2) { double s = 0; for (long long q = 0; q < n; ++q) s += w[q] * w[q]; *nrm2 = s; }
}
void gs_final(Stream*, const double* V, long long ldv, int nvec, const double* w, long long n, const double* coef, const double* nrm2_in, double* nrm2_out,
              double* vout) {
    ++g_launches;
    if (nvec > MAX_BASIS + 1) throw std::runtime_error("gs_final: nvec " + std::to_string(nvec) + " exceeds MAX_BASIS + 1");
    double s = 0;
    for (int i = 0; i < nvec; ++i) s += coef[i] * coef[i];
    const bool skip = s <= GS_REFINE_REL * GS_REFINE_REL * *nrm2_in;
    double b2 = skip ? *nrm2_in : *nrm2_in - s;
    if (!(b2 > 0.0)) b2 = 0.0;
    const double inv = b2 > 0.0 ? 1.0 / std::sqrt(b2) : 0.0;
    *nrm2_out = b2;
    for (long long q = 0; q < n; ++q) { double a = w[q]; if (!skip) for (int i = 0; i < nvec; ++i) a -= coef[i] * V[i * ldv + q]; vout[q] = a * inv; }
}
void scale_inv_norm(Stream*, const double* w, const double* nrm2, double* v, long long n) {
    ++g_launches;
    const double inv = 1.0 / std::sqrt(*nrm2);
    for (long long q = 0; q < n; ++q) v[q] = w[q] * inv;
}
void ritz_rotate(Stream*, double* V, long long ldv, long long n, int ncv, const double* S, int kk) {
    ++g_launches;
    if (ncv > MAX_BASIS + 1) throw std::runtime_error("ritz_rotate: ncv " + std::to_string(ncv) + " exceeds MAX_BASIS + 1");
    std::vector<double> v(ncv);
    for (long long q = 0; q < n; ++q) {
        for (int i = 0; i < ncv; ++i) v[i] = V[i * ldv + q];
        for (int a = 0; a < kk; ++a) { double o = 0; for (int i = 0; i < ncv; ++i) o += S[i * kk + a] * v[i]; V[a * ldv + q] = o; }
    }
}
void filter_small(Stream*, double* x, long long n, double tol) { ++g_launches; for (long long q = 0; q < n; ++q) if (std::fabs(x[q]) < tol) x[q] = 0.0; }
void axpby_out(Stream*, const double* a, const double* b, double alpha, double* out, long long n) {
    ++g_launches;
    for (long long q = 0; q < n; ++q) out[q] = (a ? a[q] : 0.0) + alpha * b[q];
}
void gather_rows_reversed(Stream*, const double* src, int n, int m, double* dst) {
    ++g_launches;
    for (int k = 0; k < m; ++k) std::memcpy(dst + (size_t)k * n, src + (size_t)(n - 1 - k) * n, sizeof(double) * n);
}
/* cyclic Jacobi; row k of A on exit = k-th eigenvector, ascending eigenvalues.  The rotations run in long double: in
   double, sequential Jacobi leaves about 2n·u·||A|| in the eigenvalues and 6n·u in the orthogonality, above what the
   eigensolver tests (tests/test_sparse_eig_kernels.py) require of syevd_batch at a few hundred states. */
static void jacobi(int n, double* A0, double* w) {
    ++g_launches;
    typedef long double R;
    std::vector<R> A(A0, A0 + (size_t)n * n), V((size_t)n * n, 0.0L);
    for (int i = 0; i < n; ++i) V[(size_t)i * n + i] = 1.0L;
    auto a = [&](int i, int j) -> R& { return A[(size_t)i * n + j]; };
    for (int sweep = 0; sweep < 100; ++sweep) {
        R off = 0, diag = 0;
        for (int i = 0; i < n; ++i) { diag += a(i, i) * a(i, i); for (int j = i + 1; j < n; ++j) off += a(i, j) * a(i, j); }
        if (off <= 1e-34L * (diag + off) || off == 0.0L) break;
        for (int p = 0; p < n; ++p)
            for (int q = p + 1; q < n; ++q) {
                if (a(p, q) == 0.0L) continue;
                R theta = (a(q, q) - a(p, p)) / (2.0L * a(p, q));
                R t = (theta >= 0 ? 1.0L : -1.0L) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0L));
                R c = 1.0L / std::sqrt(t * t + 1.0L), s = t * c;
                for (int k = 0; k < n; ++k) { R akp = a(k, p), akq = a(k, q); a(k, p) = c * akp - s * akq; a(k, q) = s * akp + c * akq; }
                for (int k = 0; k < n; ++k) { R apk = a(p, k), aqk = a(q, k); a(p, k) = c * apk - s * aqk; a(q, k) = s * apk + c * aqk; }
                for (int k = 0; k < n; ++k) { R vkp = V[(size_t)k * n + p], vkq = V[(size_t)k * n + q]; V[(size_t)k * n + p] = c * vkp - s * vkq; V[(size_t)k * n + q] = s * vkp + c * vkq; }
            }
    }
    std::vector<int> ord(n);
    for (int i = 0; i < n; ++i) ord[i] = i;
    std::vector<R> d(n);
    for (int i = 0; i < n; ++i) d[i] = a(i, i);
    std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return d[x] < d[y]; });
    for (int k = 0; k < n; ++k) { w[k] = (double)d[ord[k]]; for (int i = 0; i < n; ++i) A0[(size_t)k * n + i] = (double)V[(size_t)i * n + ord[k]]; }
}

int syevd_batch(Stream*, int nblocks, const int* n, double* const* A, double* const* w) {
    for (int b = 0; b < nblocks; ++b)
        if (n[b] > 0) jacobi(n[b], A[b], w[b]);
    return 0;
}

/* collectives of the emulation: callbacks registered by the test (tests/test_dist_cpu.py implements them with
   torch.distributed over gloo, one process per emulated GPU) */
typedef void (*allreduce_cb_t)(double* buf, long long n);
typedef void (*bcast_cb_t)(double* buf, long long n, int root);
static allreduce_cb_t g_allreduce = nullptr;
static bcast_cb_t g_bcast = nullptr;
static int g_rank = 0, g_world = 1;
int comm_unique_id(void* out) { std::memset(out, 0, COMM_ID_BYTES); return 0; }
int comm_init(Stream*, int rank, int world, const void*) { g_rank = rank; g_world = world; return 0; }
void allreduce_sum(Stream*, double* buf, long long n) { if (g_world > 1 && n > 0) g_allreduce(buf, n); }
void allgatherv(Stream*, double* buf, const long long* off) {
    if (g_world <= 1) return;
    for (int r = 0; r < g_world; ++r) if (off[r + 1] > off[r]) g_bcast(buf + off[r], off[r + 1] - off[r], r);
}
/* delivered to the named receiver ONLY (the other ranks take the broadcast into a scratch buffer): a halo the planner forgot
   stays missing and the parity tests see it */
void exchange_ranges(Stream*, double* buf, int n, const int* from, const int* to, const long long* off, const long long* cnt) {
    if (g_world <= 1) return;
    std::vector<double> tmp;
    for (int i = 0; i < n; ++i) {
        if (cnt[i] <= 0 || from[i] == to[i]) continue;
        if (g_rank == from[i] || g_rank == to[i]) g_bcast(buf + off[i], cnt[i], from[i]);
        else { tmp.resize((size_t)cnt[i]); g_bcast(tmp.data(), cnt[i], from[i]); }
    }
}
void bcast_batch(Stream*, int n, double* const* ptr, const long long* count, const int* root) {
    if (g_world <= 1) return;
    for (int i = 0; i < n; ++i) if (count[i] > 0) g_bcast(ptr[i], count[i], root[i]);
}

}  // namespace dev
/* the chain plan check on its own, for a test of a plan that no buffer of a test could hold: 0, or -1 with the message */
extern "C" int plancheck_check_chain(const void* items, int nitems, const void* segs, char* msg, int len) {
    try {
        dev::check_chain_plan((const dev::WorkItem*)items, nitems, (const dev::Segment*)segs);
        return 0;
    } catch (const std::exception& e) {
        std::snprintf(msg, (size_t)len, "%s", e.what());
        return -1;
    }
}
extern "C" void plancheck_set_collectives(void (*allreduce)(double*, long long), void (*bcast)(double*, long long, int)) {
    dev::g_allreduce = allreduce;
    dev::g_bcast = bcast;
}
