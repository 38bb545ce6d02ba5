/*  dev_cuda.cu — hand-written sm_100a kernels behind dev.h.
 *
 *  chain_kernel — the one compute engine of the path (H·psi stages 1 and 2, rho = X·Xᵀ, O·Uᵀ, U·T, enlarged H, operator
 *  products).  One CTA per ≤64×64 output tile, 4 warps in a 2×2 grid, each warp up to a 32×32 sub-tile held as 4×4 FP64 DMMA
 *  (mma.sync.m8n8k4.f64) accumulator fragments; a tile accumulates its whole chain of segments in registers and is written
 *  once.  Operand chunks of 16 in K are staged global→shared with cp.async (LDGSTS.64, K tail by the zero-fill size operand,
 *  rows of ragged tiles clamped), double-buffered; the shared layouts are padded (row stride ≡ 4 mod 16 doubles) so that both
 *  the row-major and the transposed fragment reads are bank-conflict-free, and the layouts are template parameters so every
 *  LDS offset is an immediate.  FP64 has no tcgen05/UMMA kind, so DMMA through mma.sync is the Blackwell tensor path for
 *  this arithmetic (SURVEY.md §7).  A predicated-off DMMA still occupies the tensor pipe for its 16 cycles, so ragged tiles
 *  dispatch per chunk to a body compiled for exactly the warp's fragment counts (profiles/r1_chain_kernel.md).
 *  Sparse (CSR), AXPY and scaled-identity factors are accumulated into the same register tile by slow-path segments.
 *
 *  Also here: gs_pass_kernel (fused Gram-Schmidt passes of the Lanczos solver, HBM-bound, deterministic last-block
 *  reductions), spmm_kernel (the sparse-sector matvec of un-truncated blocks, TMA-staged), the batched eigensolvers of the
 *  reduced-density-matrix blocks (jacobi_eig_kernel up to 64 states, block Jacobi with DMMA updates above), the NCCL
 *  collectives (bound lazily) and the slab-based caching allocator.  No vendor math library is linked.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>

#include <chrono>
#include <map>
#include <unordered_map>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <stdexcept>
#include <string>
#include <vector>

#include "dev.h"

namespace dev {

static thread_local std::string g_err;
static long long g_launches = 0;
const char* last_error() { return g_err.c_str(); }
long long launch_count() { return g_launches; }

#define CUDA_OK(call)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            char buf_[512];                                                                             \
            snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
            g_err = buf_;                                                                               \
            fprintf(stderr, "[dmrgx] %s\n", buf_);                                                      \
            throw std::runtime_error(buf_);                                                             \
        }                                                                                               \
    } while (0)

struct Stream {
    int device = 0;
    cudaStream_t s = nullptr;
    bool own = false;
    double* partials = nullptr; /* deterministic two-stage reductions */
    unsigned int* ticket = nullptr; /* "last block finishes the reduction" counter of gs_pass */
    int num_sms = 148;
    struct Arena { char* base = nullptr; size_t size = 0; std::map<size_t, size_t> free; /* offset -> length of the free ranges */ };
    std::vector<Arena> arenas;   /* what was actually cudaMalloc'ed */
    std::unordered_map<void*, size_t> live;
    size_t bytes_reserved = 0, bytes_free = 0, bytes_live = 0, bytes_live_peak = 0;
    double malloc_seconds = 0;   /* time spent in cudaMalloc for the heap (DMRGX_TRACE / DMRGX_ALLOC_STATS print it at the end) */
    long long malloc_calls = 0;
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    int spmm_smem = 0;           /* dynamic shared memory spmm_kernel has been configured for on this device */
    bool chain_cfg = false;      /* chain_kernel's dynamic shared memory attribute has been set on this device */
    bool gram_cfg = false;       /* the same for gram_kernel */
    bool gram_rect_cfg = false;  /* the same for gram_kernel<true> (gram_rect) */
    cudaStream_t aux = nullptr;  /* side stream: the small-block eigensolver runs beside the block-Jacobi launches */
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

constexpr int RED_BLOCKS = 592; /* 148 SMs × 4 resident CTAs */
constexpr int RED_MAXVEC = 40;

int init(int device, void* user_stream, Stream** out) {
    try {
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0) {
            g_err = std::string("no CUDA device: ") + cudaGetErrorString(e) + " — dmrgx has no CPU path";
            return 100;
        }
        CUDA_OK(cudaSetDevice(device));
        Stream* st = new Stream();
        st->device = device;
        if (user_stream) { st->s = (cudaStream_t)user_stream; st->own = false; }
        else { CUDA_OK(cudaStreamCreateWithFlags(&st->s, cudaStreamNonBlocking)); st->own = true; }
        cudaDeviceProp prop;
        CUDA_OK(cudaGetDeviceProperties(&prop, device));
        st->num_sms = prop.multiProcessorCount;
        CUDA_OK(cudaMalloc(&st->partials, sizeof(double) * RED_BLOCKS * RED_MAXVEC));
        CUDA_OK(cudaMalloc(&st->ticket, sizeof(unsigned int)));
        CUDA_OK(cudaMemset(st->ticket, 0, sizeof(unsigned int)));
        *out = st;
        return 0;
    } catch (const std::exception&) { return 100; }
}

static void comm_destroy_(Stream* st);
void destroy(Stream* st) {
    if (!st) return;
    cudaSetDevice(st->device);
    cudaStreamSynchronize(st->s);
    if (getenv("DMRGX_TRACE") || getenv("DMRGX_ALLOC_STATS"))
        fprintf(stderr, "[trace] allocator: %lld cudaMalloc calls, %.3f s, %.2f GB reserved, peak in use %.2f GB\n", st->malloc_calls, st->malloc_seconds,
                st->bytes_reserved / 1e9, st->bytes_live_peak / 1e9);
    if (st->comm) comm_destroy_(st);
    if (st->aux) cudaStreamDestroy(st->aux);
    if (st->ev_fork) cudaEventDestroy(st->ev_fork);
    if (st->ev_join) cudaEventDestroy(st->ev_join);
    for (auto& ar : st->arenas) cudaFree(ar.base);
    cudaFree(st->partials);
    cudaFree(st->ticket);
    if (st->own) cudaStreamDestroy(st->s);
    delete st;
}
void make_current(Stream* st) { cudaSetDevice(st->device); }

/* Device memory: a stream-ordered heap.  A DMRG sweep frees and allocates panels of slowly varying sizes every step; handing
   each one back to the driver (cudaFreeAsync) let the pool fragment and re-map (200-700 ms stalls inside single steps), and
   round 1's size-class free lists reserved 65 GB for a 12x6 m = 2048 run once the eigensolver workspaces joined the mix
   (profiles/r2_eigensolver.md).  Now: arenas of 1-8 GiB from cudaMalloc, inside them a classic best-fit heap with splitting
   and coalescing of free ranges.  Everything is ordered on the one stream of the context, so a freed range can be handed out
   again immediately: its new user is queued behind its old one. */
constexpr size_t HEAP_SLAB = (size_t)1 << 30, HEAP_GRAIN = (size_t)256 << 20;
static void heap_add_arena(Stream* st, void* slab, size_t sz) {
    Stream::Arena ar; ar.base = (char*)slab; ar.size = sz; ar.free[0] = sz;
    st->arenas.push_back(ar); st->bytes_reserved += sz; st->bytes_free += sz;
}
void* malloc_bytes(Stream* st, size_t bytes) {
    const size_t need = (std::max<size_t>(bytes, 1) + 511) & ~(size_t)511;
    for (;;) {
        /* best fit over the free ranges of all arenas */
        Stream::Arena* best_a = nullptr;
        std::map<size_t, size_t>::iterator best;
        size_t best_len = ~(size_t)0;
        for (auto& ar : st->arenas)
            for (auto f = ar.free.begin(); f != ar.free.end(); ++f)
                if (f->second >= need && f->second < best_len) { best_a = &ar; best = f; best_len = f->second; if (best_len == need) break; }
        if (best_a) {
            const size_t off = best->first, len = best->second;
            best_a->free.erase(best);
            if (len > need) best_a->free[off + need] = len - need;
            void* p = best_a->base + off;
            st->live[p] = need;
            st->bytes_free -= need; st->bytes_live += need;
            if (st->bytes_live > st->bytes_live_peak) st->bytes_live_peak = st->bytes_live;
            return p;
        }
        /* a new arena: 1 GiB, a quarter of what is already reserved (at most 8 GiB: the 0.4-1.5 GB blocks and workspaces of a
           large sweep pack poorly into 1 GiB arenas — 53 GB reserved for 37 GB in use on the 12x6 m = 2048 run), or the
           request rounded up to 256 MiB when larger */
        const size_t quarter = std::min(HEAP_SLAB * 8, st->bytes_reserved / 4 / HEAP_GRAIN * HEAP_GRAIN);
        const size_t sz = std::max(std::max(HEAP_SLAB, quarter), (need + HEAP_GRAIN - 1) / HEAP_GRAIN * HEAP_GRAIN);
        void* slab = nullptr;
        const auto t0 = std::chrono::steady_clock::now();
        cudaError_t e = cudaMalloc(&slab, sz);
        if (e != cudaSuccess) {
            /* out of memory: give wholly free arenas back to the driver and try once more (with just what is needed) */
            cudaGetLastError();
            CUDA_OK(cudaStreamSynchronize(st->s));
            for (size_t i = 0; i < st->arenas.size();) {
                Stream::Arena& ar = st->arenas[i];
                if (ar.free.size() == 1 && ar.free.begin()->second == ar.size) {
                    cudaFree(ar.base); st->bytes_reserved -= ar.size; st->bytes_free -= ar.size; st->arenas.erase(st->arenas.begin() + (long)i);
                } else ++i;
            }
            e = cudaMalloc(&slab, need);
            if (e == cudaSuccess) heap_add_arena(st, slab, need);
        } else heap_add_arena(st, slab, sz);
        st->malloc_seconds += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        st->malloc_calls++;
        CUDA_OK(e); /* throws when the device is full; otherwise the new arena holds the request and the next pass returns */
    }
}
void free_bytes(Stream* st, void* p) {
    if (!p) return;
    auto f = st->live.find(p);
    if (f == st->live.end()) return;
    size_t len = f->second;
    st->live.erase(f);
    st->bytes_free += len; st->bytes_live -= len;
    for (auto& ar : st->arenas) {
        if ((char*)p < ar.base || (char*)p >= ar.base + ar.size) continue;
        size_t off = (size_t)((char*)p - ar.base);
        auto nx = ar.free.lower_bound(off);
        if (nx != ar.free.end() && off + len == nx->first) { len += nx->second; nx = ar.free.erase(nx); } /* merge with the next range */
        if (nx != ar.free.begin()) {
            auto pv = std::prev(nx);
            if (pv->first + pv->second == off) { pv->second += len; return; }                             /* ... and the previous one */
        }
        ar.free[off] = len;
        return;
    }
}
void h2d(Stream* st, void* dst, const void* src, size_t bytes) { if (bytes) CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st->s)); }
void d2h(Stream* st, void* dst, const void* src, size_t bytes) { if (bytes) CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st->s)); }
void d2d(Stream* st, void* dst, const void* src, size_t bytes) { if (bytes) CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st->s)); }
void memset0(Stream* st, void* dst, size_t bytes) { if (bytes) CUDA_OK(cudaMemsetAsync(dst, 0, bytes, st->s)); }
void sync(Stream* st) { CUDA_OK(cudaStreamSynchronize(st->s)); }

#define LAUNCH_CHECK() do { ++g_launches; CUDA_OK(cudaGetLastError()); } while (0)

/* ================================================================================================
 *  chain_kernel
 * ============================================================================================== */
constexpr int BM = 64, BK = 16, NTHREADS = 128;
constexpr int S_MK = BK + 4;  /* [m][k] layout row stride (20 ≡ 4 mod 16) */
constexpr int S_KM = BM + 4;  /* [k][m] layout row stride (68 ≡ 4 mod 16) */
constexpr int SMEM_TILE = (BM * S_MK > BK * S_KM) ? BM * S_MK : BK * S_KM; /* 1280 doubles */
/* NSTAGE (template parameter of the kernel): depth of the cp.async ring — chunks c+1 .. c+NSTAGE-1 are in flight while chunk c is
   multiplied.  Two stages are best when the launch is large and its operands are L2-warm (m = 2048: 1.264 vs 1.294 ms); three win
   when the work items are few and every operand is a cold DRAM miss (one rank's shard of an 8-GPU apply: stage 2 0.158 -> 0.121 ms):
   run_chain picks by the size of the launch (profiles/r2_chain_kernel.md). */

__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gsrc, bool valid) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async8_all(double* smem_dst, const double* gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

/* ---- operand staging ------------------------------------------------------------------------
 *  Each thread owns 8 elements of the A chunk and 8 of the B chunk.  Rows beyond the tile extent are
 *  CLAMPED to the last valid row (their products land in accumulator rows that are never stored), so
 *  the only predicate is the K tail — carried by the zero-fill size operand of cp.async, one code path —
 *  and the global pointers are bumped by a constant per chunk.  Layout template parameters make every
 *  shared-memory offset an immediate.                                                             */
template <bool MK> /* MK: operand contiguous along k -> smem [row][k]; else contiguous along row -> smem [k][row] */
struct Stager {
    const double* base;  /* bumped by kstep per chunk */
    int off[8];          /* element offsets of this thread's 8 elements (rows clamped to the tile extent) */
    long long kstep;     /* pointer advance per chunk, in elements */
    int soff;            /* smem offset of element 0; element i is at soff + i*SI */
    int k0;              /* k index of element 0 inside a chunk (element i: k0 for MK, k0 + 2i otherwise) */
    unsigned rowmask;    /* bit i: element i lies in a row of the tile (rows beyond a ragged tile's extent are not staged at all:
                            their shared-memory lines keep stale data that only reaches accumulator rows / columns never stored) */
    static constexpr int SI = MK ? 8 * S_MK : 2 * S_KM;
    __device__ __forceinline__ void init(const double* b, long long ld_row, long long ld_k, int ext, int tid) {
        base = b;
        if (MK) {
            const int k = tid & 15, r0 = tid >> 4;
            rowmask = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                int r = r0 + 8 * i;
                if (r < ext) rowmask |= 1u << i;
                r = r < ext ? r : ext - 1;
                off[i] = (int)(r * ld_row + k * ld_k);
            }
            soff = r0 * S_MK + k;
            k0 = k;
        } else {
            const int r = tid & 63, kk = tid >> 6;
            const int rc = r < ext ? r : ext - 1;
            rowmask = r < ext ? 0xffu : 0u;
#pragma unroll
            for (int i = 0; i < 8; ++i) off[i] = (int)(rc * ld_row + (kk + 2 * i) * ld_k);
            soff = kk * S_KM + r;
            k0 = kk;
        }
        kstep = (long long)BK * ld_k;
    }
    /* krem = K - k0 of this chunk (>= 1); ALLROWS: a full tile, no row is skipped */
    template <bool ALLROWS>
    __device__ __forceinline__ void issue(double* sm, int krem) {
        if (krem >= BK) { /* block-uniform: every chunk but a segment's last one — no K predicate, no pointer select */
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (ALLROWS || ((rowmask >> i) & 1u)) cp_async8_all(sm + soff + i * SI, base + off[i]);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const bool v = (MK ? k0 : k0 + 2 * i) < krem;
                if (ALLROWS || ((rowmask >> i) & 1u)) cp_async8(sm + soff + i * SI, v ? base + off[i] : base, v);
            }
        }
        base += kstep;
    }
};

/* One GEMM segment of a chain.  FULL: a 64×64 tile with a unit coefficient — every warp owns 4×4 fragments, no predicate
   and no multiply in the inner loop (the plan folds the couplings into the right factors, so this is where the flops
   are).  Otherwise the generic variant: fragment counts and the coefficient are runtime values.  Two variants per
   operand layout keep the kernel small enough for the instruction caches. */
/* the DMMAs of one 16-deep chunk for a warp that owns NMI x NNI fragments */
template <bool A_MK, bool B_NK, bool UNIT, int NMI, int NNI, int NKK = BK / 4>
__device__ __forceinline__ void chunk_mma(double (&acc)[4][4][2], const double* as, const double* bs, double coef) {
    constexpr int a_sm = A_MK ? S_MK : 1, a_sk = A_MK ? 1 : S_KM;
    constexpr int b_sn = B_NK ? S_MK : 1, b_sk = B_NK ? 1 : S_KM;
#pragma unroll
    for (int kk = 0; kk < NKK; ++kk) {
        double a[NMI], b[NNI];
#pragma unroll
        for (int mi = 0; mi < NMI; ++mi) a[mi] = as[mi * 8 * a_sm + kk * 4 * a_sk];
#pragma unroll
        for (int ni = 0; ni < NNI; ++ni) b[ni] = UNIT ? bs[ni * 8 * b_sn + kk * 4 * b_sk] : bs[ni * 8 * b_sn + kk * 4 * b_sk] * coef;
#pragma unroll
        for (int ni = 0; ni < NNI; ++ni)
#pragma unroll
            for (int mi = 0; mi < NMI; ++mi) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
    }
}

template <int NSTAGE, bool A_MK, bool B_NK, bool FULL, bool UNIT>
__device__ __forceinline__ void gemm_segment(double (&acc)[4][4][2], const Segment& sg, const WorkItem& it, double* As, double* Bs,
                                             int tid, int rbase, int cbase, int g, int t, int nmi, int nni) {
    Stager<A_MK> sa;
    Stager<B_NK> sb;
    sa.init(sg.A + (long long)it.m0 * sg.lda_m, sg.lda_m, sg.lda_k, it.tm, tid);
    sb.init(sg.B + (long long)it.n0 * sg.ldb_n, sg.ldb_n, sg.ldb_k, it.tn, tid);
    const int K = sg.K;
    const int nchunks = (K + BK - 1) / BK;
    const double coef = sg.coef;
    constexpr int a_sm = A_MK ? S_MK : 1, a_sk = A_MK ? 1 : S_KM;
    constexpr int b_sn = B_NK ? S_MK : 1, b_sk = B_NK ? 1 : S_KM;
    const int a_base = (rbase + g) * a_sm + t * a_sk;
    const int b_base = (cbase + g) * b_sn + t * b_sk;
    __syncthreads(); /* the previous segment's readers are done with every stage */
    /* prologue: the first NSTAGE-1 chunks; a group is committed for every slot (empty past the end) so that the wait below
       always means "all but the NSTAGE-1 most recent groups", i.e. chunk c, have landed */
#pragma unroll
    for (int p = 0; p < NSTAGE - 1; ++p) {
        if (p < nchunks) {
            sa.template issue<FULL>(As + p * SMEM_TILE, K - p * BK);
            sb.template issue<FULL>(Bs + p * SMEM_TILE, K - p * BK);
        }
        cp_async_commit();
    }
    /* (a one-barrier-per-chunk ring — wait, barrier, then refill the stage of chunk c-1 — was measured: 0.2 % slower) */
    int cur = 0, nxt = NSTAGE - 1;
    for (int c = 0; c < nchunks; ++c) {
        if (c + NSTAGE - 1 < nchunks) {
            const int krem = K - (c + NSTAGE - 1) * BK;
            sa.template issue<FULL>(As + nxt * SMEM_TILE, krem);
            sb.template issue<FULL>(Bs + nxt * SMEM_TILE, krem);
        }
        cp_async_commit();
        cp_async_wait<NSTAGE - 1>();
        __syncthreads();
        const double* as = As + cur * SMEM_TILE + a_base;
        const double* bs = Bs + cur * SMEM_TILE + b_base;
        if (FULL) {
            /* the last chunk of a segment holds K mod 16 columns: only the 4-deep steps that contain any are run */
            const int krem = K - c * BK;
            if (krem > 12) chunk_mma<A_MK, B_NK, UNIT, 4, 4, 4>(acc, as, bs, coef);
            else if (krem > 8) chunk_mma<A_MK, B_NK, UNIT, 4, 4, 3>(acc, as, bs, coef);
            else if (krem > 4) chunk_mma<A_MK, B_NK, UNIT, 4, 4, 2>(acc, as, bs, coef);
            else chunk_mma<A_MK, B_NK, UNIT, 4, 4, 1>(acc, as, bs, coef);
        } else {
            /* ragged tile: the fragment counts of this warp select a body compiled for exactly that many DMMAs — a predicated-off
               DMMA still occupies the tensor pipe (a 32x32 tile took as long as a 64x64 one) */
#define MMA_CASE(M_, N_) case (M_) * 5 + (N_): chunk_mma<A_MK, B_NK, UNIT, M_, N_>(acc, as, bs, coef); break;
            switch (nmi * 5 + nni) {
                MMA_CASE(4, 4) MMA_CASE(4, 3) MMA_CASE(4, 2) MMA_CASE(4, 1)
                MMA_CASE(3, 4) MMA_CASE(3, 3) MMA_CASE(3, 2) MMA_CASE(3, 1)
                MMA_CASE(2, 4) MMA_CASE(2, 3) MMA_CASE(2, 2) MMA_CASE(2, 1)
                MMA_CASE(1, 4) MMA_CASE(1, 3) MMA_CASE(1, 2) MMA_CASE(1, 1)
                default: break;
            }
#undef MMA_CASE
        }
        __syncthreads();
        cur = cur + 1 == NSTAGE ? 0 : cur + 1;
        nxt = nxt + 1 == NSTAGE ? 0 : nxt + 1;
    }
}

template <int NSTAGE, bool A_MK, bool B_NK>
__device__ __forceinline__ void gemm_dispatch(double (&acc)[4][4][2], const Segment& sg, const WorkItem& it, double* As, double* Bs,
                                              int tid, int rbase, int cbase, int g, int t, int nmi, int nni) {
    /* block-uniform choice: every warp of a 64×64 tile has 4×4 fragments */
    if (sg.coef == 1.0) {
        if (it.tm == BM && it.tn == BM) gemm_segment<NSTAGE, A_MK, B_NK, true, true>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, 4, 4);
        else gemm_segment<NSTAGE, A_MK, B_NK, false, true>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, nmi, nni);
    } else gemm_segment<NSTAGE, A_MK, B_NK, false, false>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, nmi, nni);
}

template <int NSTAGE>
__global__ void __launch_bounds__(NTHREADS, 3) chain_kernel(const WorkItem* __restrict__ items, const Segment* __restrict__ segs,
                                                            const double* __restrict__ xbase, double* __restrict__ ybase,
                                                            double* __restrict__ wbase) {
    extern __shared__ __align__(16) double chain_smem[];
    double* As = chain_smem;
    double* Bs = chain_smem + NSTAGE * SMEM_TILE;
    WorkItem it = items[blockIdx.x];
    if (it.c_in_y) it.C = (double*)((char*)(it.c_in_y == 1 ? ybase : wbase) + (size_t)it.C);
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int wm = warp >> 1, wn = warp & 1;
    const int g = lane >> 2, t = lane & 3;
    const int tm = it.tm, tn = it.tn;
    /* the tile is split evenly between the two warp rows / columns (plan.cpp makes extents multiples of 16 except at
       the ragged edge): rows [rbase, rbase + 8*nmi) and columns [cbase, cbase + 8*nni) belong to this warp */
    const int hm = ((tm + 15) >> 4) << 3, hn = ((tn + 15) >> 4) << 3;
    const int rbase = wm * hm, cbase = wn * hn;
    int nmi = (tm - rbase + 7) / 8; nmi = nmi < 0 ? 0 : (nmi > (hm >> 3) ? (hm >> 3) : nmi);
    int nni = (tn - cbase + 7) / 8; nni = nni < 0 ? 0 : (nni > (hn >> 3) ? (hn >> 3) : nni);

    double acc[4][4][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }

    for (int s = it.seg_begin; s < it.seg_end; ++s) {
        Segment sg = segs[s];
        if (sg.flags & SEGF_A_X) sg.A = (const double*)((const char*)xbase + (size_t)sg.A);
        if (sg.flags & SEGF_B_X) sg.B = (const double*)((const char*)xbase + (size_t)sg.B);
        if (sg.type == SEG_GEMM) {
            const bool a_mk = (sg.lda_k == 1) || (sg.lda_m != 1);
            const bool b_nk = (sg.ldb_k == 1) || (sg.ldb_n != 1);
            if (a_mk) {
                if (b_nk) gemm_dispatch<NSTAGE, true, true>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, nmi, nni);
                else gemm_dispatch<NSTAGE, true, false>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, nmi, nni);
            } else {
                if (b_nk) gemm_dispatch<NSTAGE, false, true>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, nmi, nni);
                else gemm_dispatch<NSTAGE, false, false>(acc, sg, it, As, Bs, tid, rbase, cbase, g, t, nmi, nni);
            }
        } else if (sg.type == SEG_AXPY) {
            /* acc += coef * A(m,n): all of a thread's (up to 32) loads are issued before the first use */
            const double* base = sg.A + (long long)(it.m0 + rbase + g) * sg.lda_m + (long long)(it.n0 + cbase + 2 * t) * sg.lda_k;
            const long long sm8 = 8 * sg.lda_m, sn8 = 8 * sg.lda_k, sn1 = sg.lda_k;
            double v[4][4][2];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const bool rok = mi < nmi && rbase + mi * 8 + g < tm;
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) {
                    const int col = cbase + ni * 8 + 2 * t;
                    const bool c0 = rok && ni < nni && col < tn, c1 = rok && ni < nni && col + 1 < tn;
                    const double* q = base + mi * sm8 + ni * sn8;
                    v[mi][ni][0] = c0 ? q[0] : 0.0;
                    v[mi][ni][1] = c1 ? q[sn1] : 0.0;
                }
            }
            const double coef = sg.coef;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) { acc[mi][ni][0] += coef * v[mi][ni][0]; acc[mi][ni][1] += coef * v[mi][ni][1]; }
        } else if (sg.type == SEG_CSRA) {
            /* sparse left factor: acc(m,n) += coef * Σ_e val[e] · X(col[e], n).  One walk over the CSR row per accumulator ROW:
               the index and value of an entry are loaded once and feed the eight columns this thread owns (the four lanes of a
               quad read 64 contiguous bytes of the dense row), instead of one dependent walk per element */
            const double* xb = sg.A + (long long)(it.n0 + cbase + 2 * t) * sg.ldb_n;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int row = rbase + mi * 8 + g;
                if (mi >= nmi || row >= tm) continue;
                const int r = sg.row0 + it.m0 + row;
                const int e1 = sg.rowptr[r + 1];
                for (int e = sg.rowptr[r]; e < e1; ++e) {
                    const double v = sg.B[e] * sg.coef;
                    const double* xr = xb + (long long)sg.colidx[e] * sg.ldb_k;
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) {
                        const int col = cbase + ni * 8 + 2 * t;
                        if (ni < nni && col < tn) acc[mi][ni][0] += v * xr[(long long)(ni * 8) * sg.ldb_n];
                        if (ni < nni && col + 1 < tn) acc[mi][ni][1] += v * xr[(long long)(ni * 8 + 1) * sg.ldb_n];
                    }
                }
            }
        } else if (sg.type == SEG_CSRB) {
            /* sparse right factor: acc(m,n) += coef * Σ_e val_n[e] · V(m, col_n[e]): one walk per accumulator COLUMN feeding the
               four rows this thread owns (lock-step walks of the eight columns were measured: no gain, the segment is bound by L2
               gather traffic, not by the length of the dependent chains) */
            const double* vb = sg.A + (long long)(it.m0 + rbase + g) * sg.lda_m;
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int col = cbase + ni * 8 + 2 * t + h;
                    if (ni >= nni || col >= tn) continue;
                    const int r = sg.row0 + it.n0 + col;
                    const int e1 = sg.rowptr[r + 1];
                    for (int e = sg.rowptr[r]; e < e1; ++e) {
                        const double v = sg.B[e] * sg.coef;
                        const double* vc = vb + (long long)sg.colidx[e] * sg.lda_k;
#pragma unroll
                        for (int mi = 0; mi < 4; ++mi)
                            if (mi < nmi && rbase + mi * 8 + g < tm) acc[mi][ni][h] += v * vc[(long long)(mi * 8) * sg.lda_m];
                    }
                }
            }
        } else if (sg.type == SEG_CSRADD) {
            /* acc(m,n) += coef * Σ_e val[e] · [col[e] == n + d]: one walk per row, each entry lands in at most one owned column */
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int row = rbase + mi * 8 + g;
                if (mi >= nmi || row >= tm) continue;
                const int r = sg.row0 + it.m0 + row;
                const int e1 = sg.rowptr[r + 1];
                for (int e = sg.rowptr[r]; e < e1; ++e) {
                    const int lc = sg.colidx[e] - sg.d - it.n0 - cbase - 2 * t; /* column relative to this thread's first one */
                    const double v = sg.B[e] * sg.coef;
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) {
                        const int col = cbase + ni * 8 + 2 * t;
                        if (ni < nni && lc == ni * 8 && col < tn) acc[mi][ni][0] += v;
                        if (ni < nni && lc == ni * 8 + 1 && col + 1 < tn) acc[mi][ni][1] += v;
                    }
                }
            }
        } else if (sg.type == SEG_DIAG) {
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int row = rbase + mi * 8 + g;
                if (mi >= nmi || row >= tm) continue;
#pragma unroll
                for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int col = cbase + ni * 8 + 2 * t + h;
                        if (ni < nni && col < tn && it.m0 + row + sg.d == it.n0 + col) acc[mi][ni][h] += sg.coef;
                    }
            }
        }
    }
    /* epilogue: each element written exactly once */
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
        const int row = rbase + mi * 8 + g;
        if (mi >= nmi || row >= tm) continue;
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int col = cbase + ni * 8 + 2 * t + h;
                if (ni >= nni || col >= tn) continue;
                double* p = it.C + (long long)row * it.ldc + col;
                if (it.mode == 0) *p = acc[mi][ni][h];
                else atomicAdd(p, acc[mi][ni][h]);
            }
        }
    }
}

void run_chain(Stream* st, const WorkItem* d_items, int nitems, const Segment* d_segs, const double* x, double* y, double* w) {
    if (nitems <= 0) return;
    constexpr int smem2 = 2 * 2 * SMEM_TILE * (int)sizeof(double), smem3 = 2 * 3 * SMEM_TILE * (int)sizeof(double);
    if (!st->chain_cfg) { /* a per-device attribute, set once per context */
        CUDA_OK(cudaFuncSetAttribute(chain_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem3));
        st->chain_cfg = true;
    }
    /* fewer than four waves of the 444 resident CTAs: the deeper copy ring (cold operands, short items) */
    constexpr int deep_below = 1800;
    if (nitems < deep_below) chain_kernel<3><<<nitems, NTHREADS, smem3, st->s>>>(d_items, d_segs, x, y, w);
    else chain_kernel<2><<<nitems, NTHREADS, smem2, st->s>>>(d_items, d_segs, x, y, w);
    LAUNCH_CHECK();
}

/* ================================================================================================
 *  spmm_kernel — the sparse-sector matvec (north_star (a)): un-truncated blocks, every operator factor sparse or the
 *  identity.  One CTA per (sector pair, SP_ROWS = 4 consecutive left rows); threads run along the right index and keep all
 *  SP_ROWS rows of their (strided) columns in registers, so every access to psi is a coalesced row segment, a right
 *  factor's (column, value) pair is fetched once and used for eight rows, and y is written exactly once.
 *    - the CTA's own rows of X_p (one contiguous range of psi) are staged in shared memory by ONE TMA bulk copy
 *      (cp.async.bulk + mbarrier; a leading / trailing element is patched by hand when the range is not 16-byte aligned);
 *      every right-factor gather X[l, col(f)] (1⊗H_R, Sz⊗Sz, ...) and every left-factor entry that falls inside the tile
 *      (the diagonal and the short-range part of H_L) is then served from shared memory;
 *    - left-factor entries outside the tile read whole rows of X_q from L2 (psi fits in L2: DRAM sees it once); the row
 *      programs are slot-major (k-th entry of each of the eight rows together), so 16 independent coalesced loads per thread
 *      are in flight before the first FMA;
 *    - right factors are slot-major ELL over the output columns: coalesced, branch-free reads, no row-pointer indirection;
 *    - the tile's program (terms x left-factor entries, flattened at plan time) is fetched into shared memory while the TMA
 *      copy is in flight; all terms accumulate in registers; one launch per apply.
 * ============================================================================================== */
constexpr int SP_BD = 256, SP_CH = 4, SP_AMAX = 24, SP_BMAX = 8;

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* b, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(b)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* b, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(b))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* b, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(ok) : "r"(smem_u32(b)), "r"(parity) : "memory");
    } while (!ok);
}

/* stage `count` records of `bytes` each from global into a shared array (all threads) */
template <class T>
__device__ __forceinline__ void sp_stage(T* dst, const T* src, int count, int tid) {
    for (int i = tid; i < count * (int)(sizeof(T) / 8); i += SP_BD) ((double*)dst)[i] = __ldg((const double*)src + i);
}

__global__ void __launch_bounds__(SP_BD, 3) spmm_kernel(const SpTile* __restrict__ tiles, const SpASlot* __restrict__ aslots, const SpSSlot* __restrict__ sslots,
                                                       const SpBSlot* __restrict__ bslots, const double* __restrict__ x, double* __restrict__ y) {
    extern __shared__ __align__(16) unsigned char sp_smem[];
    __shared__ unsigned long long mbar;
    __shared__ SpTile s_tile;
    __shared__ SpASlot s_a[SP_AMAX];
    __shared__ SpSSlot s_s[SP_AMAX];
    __shared__ SpBSlot s_b[SP_BMAX];
    const int tid = threadIdx.x;
    if (tid < (int)(sizeof(SpTile) / 4)) ((int*)&s_tile)[tid] = ((const int*)(tiles + blockIdx.x))[tid];
    if (tid == 0) mbar_init(&mbar, 1);
    __syncthreads();
    const int nR = s_tile.nR, nrows = s_tile.nrows;
    const long long off0 = s_tile.off;
    /* ---- stage the tile's own rows: nrows*nR contiguous doubles of psi ---- */
    const double* src0 = x + off0;
    const int cnt = nrows * nR;
    const int head = (int)(((unsigned long long)src0 >> 3) & 1ull);   /* 1: the range starts 8 mod 16 */
    double* xs = (double*)sp_smem + head;                               /* xs + head is 16-byte aligned */
    const int bulk = (cnt - head) & ~1;
    if (tid == 0 && bulk > 0) {
        mbar_expect_tx(&mbar, (unsigned)bulk * 8u);
        bulk_g2s(xs + head, src0 + head, (unsigned)bulk * 8u, &mbar);
    }
    if (tid == 32 && head) xs[0] = src0[0];
    if (tid == 64 && head + bulk < cnt) xs[cnt - 1] = src0[cnt - 1];
    const int na = s_tile.a_count, ns = s_tile.s_count, nb = s_tile.b_count;
    bool staged = false;

    for (int cb0 = 0; cb0 < nR; cb0 += SP_CH * SP_BD) {
        double acc[SP_CH][SP_ROWS];
#pragma unroll
        for (int j = 0; j < SP_CH; ++j)
#pragma unroll
            for (int r = 0; r < SP_ROWS; ++r) acc[j][r] = 0.0;
        const int c0 = cb0 + tid;
        bool cok[SP_CH];
#pragma unroll
        for (int j = 0; j < SP_CH; ++j) cok[j] = c0 + j * SP_BD < nR;

        /* ---- identity on the right, source rows in L2: acc(r, c) += w_r · X_q(s_r, c); these loads go out first, the
                shared-memory stage is awaited only afterwards ---- */
        for (int a0 = 0; a0 < na; a0 += SP_AMAX) {
            const int nbatch = min(SP_AMAX, na - a0);
            __syncthreads(); /* the previous batch has been consumed */
            sp_stage(s_a, aslots + s_tile.a_begin + a0, nbatch, tid);
            __syncthreads();
            for (int k = 0; k < nbatch; ++k) {
#pragma unroll
                for (int h = 0; h < SP_ROWS; h += 4) {
                    double v[4][SP_CH];
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const double* p = x + s_a[k].src[h + r] + c0;
#pragma unroll
                        for (int j = 0; j < SP_CH; ++j) v[r][j] = cok[j] ? __ldg(p + j * SP_BD) : 0.0;
                    }
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const double w = s_a[k].w[h + r];
#pragma unroll
                        for (int j = 0; j < SP_CH; ++j) acc[j][h + r] += w * v[r][j];
                    }
                }
            }
        }
        if (!staged) { if (bulk > 0) mbar_wait(&mbar, 0); staged = true; }
        /* ---- the same with source rows inside the tile (the diagonal and the short-range part of H_L): shared memory ---- */
        for (int a0 = 0; a0 < ns; a0 += SP_AMAX) {
            const int nbatch = min(SP_AMAX, ns - a0);
            __syncthreads();
            sp_stage(s_s, sslots + s_tile.s_begin + a0, nbatch, tid);
            __syncthreads();
            for (int k = 0; k < nbatch; ++k) {
#pragma unroll
                for (int r = 0; r < SP_ROWS; ++r) {
                    const double* p = xs + s_s[k].roff[r] + c0;
                    const double w = s_s[k].w[r];
#pragma unroll
                    for (int j = 0; j < SP_CH; ++j)
                        if (cok[j]) acc[j][r] += w * p[j * SP_BD];
                }
            }
        }
        /* ---- right factors: acc(r, c) += w_r · Σ_t B(c, t) · X_q(s_r, col_t(c)); B(c, t) is read once for the eight rows ---- */
        for (int b0 = 0; b0 < nb; b0 += SP_BMAX) {
            const int nbatch = min(SP_BMAX, nb - b0);
            __syncthreads();
            sp_stage(s_b, bslots + s_tile.b_begin + b0, nbatch, tid);
            __syncthreads();
            for (int k = 0; k < nbatch; ++k) {
                const int W = s_b[k].W, ld = s_b[k].ld;
                const int* ecol = s_b[k].ecol + c0;
                const double* eval = s_b[k].eval + c0;
                if (s_b[k].all_in) {
                    /* every source row is one of the tile's own (1⊗H_R, Sz⊗Sz, ...): gathers from shared memory, 32-bit offsets */
#pragma unroll
                    for (int h = 0; h < SP_ROWS; h += 4) {
                        int roff[4];
                        double w[4];
#pragma unroll
                        for (int r = 0; r < 4; ++r) { roff[r] = s_b[k].roff[h + r]; w[r] = s_b[k].w[h + r]; }
                        for (int t = 0; t < W; ++t) {
                            int cf[SP_CH];
                            double vb[SP_CH];
#pragma unroll
                            for (int j = 0; j < SP_CH; ++j) {
                                cf[j] = cok[j] ? __ldg(ecol + t * ld + j * SP_BD) : 0;
                                vb[j] = cok[j] ? __ldg(eval + t * ld + j * SP_BD) : 0.0;
                            }
#pragma unroll
                            for (int j = 0; j < SP_CH; ++j) {
                                if (vb[j] == 0.0) continue; /* padding slot: no gather */
#pragma unroll
                                for (int r = 0; r < 4; ++r) acc[j][h + r] += (w[r] * vb[j]) * xs[roff[r] + cf[j]];
                            }
                        }
                    }
                } else {
#pragma unroll
                    for (int h = 0; h < SP_ROWS; h += 4) {
                        const double* gx[4];
                        double w[4];
#pragma unroll
                        for (int r = 0; r < 4; ++r) { gx[r] = x + s_b[k].src[h + r]; w[r] = s_b[k].w[h + r]; }
                        for (int t = 0; t < W; ++t) {
                            int cf[SP_CH];
                            double vb[SP_CH];
#pragma unroll
                            for (int j = 0; j < SP_CH; ++j) {
                                cf[j] = cok[j] ? __ldg(ecol + t * ld + j * SP_BD) : 0;
                                vb[j] = cok[j] ? __ldg(eval + t * ld + j * SP_BD) : 0.0;
                            }
#pragma unroll
                            for (int j = 0; j < SP_CH; ++j) {
                                if (vb[j] == 0.0) continue;
#pragma unroll
                                for (int r = 0; r < 4; ++r) acc[j][h + r] += (w[r] * vb[j]) * __ldg(gx[r] + cf[j]);
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < SP_ROWS; ++r) {
            if (r >= nrows) continue;
            double* yr = y + off0 + (long long)r * nR + c0;
#pragma unroll
            for (int j = 0; j < SP_CH; ++j)
                if (cok[j]) yr[j * SP_BD] = acc[j][r];
        }
    }
}

void run_spmm(Stream* st, const SpTile* d_tiles, int ntiles, const SpASlot* d_aslots, const SpSSlot* d_sslots, const SpBSlot* d_bslots, const double* x, double* y,
              int max_nR) {
    if (ntiles <= 0) return;
    if (max_nR > SP_MAX_NR) throw std::runtime_error("run_spmm: right sector too wide for the shared-memory stage");
    const int smem = SP_ROWS * max_nR * 8 + 32;
    if (smem > st->spmm_smem) { /* a per-device attribute, raised once per context */
        CUDA_OK(cudaFuncSetAttribute(spmm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        st->spmm_smem = smem;
    }
    spmm_kernel<<<ntiles, SP_BD, smem, st->s>>>(d_tiles, d_aslots, d_sslots, d_bslots, x, y);
    LAUNCH_CHECK();
}

__global__ void __launch_bounds__(256) reduce_kernel(const ReduceItem* __restrict__ items, double* __restrict__ ybase, const double* __restrict__ wbase) {
    const ReduceItem it = items[blockIdx.x];
    double* dst = it.dst_in_y ? (double*)((char*)ybase + (size_t)it.dst) : it.dst;
    const double* src = (const double*)((const char*)wbase + it.src_off);
    const int cnt = it.tm * it.tn;
    for (int e = threadIdx.x; e < cnt; e += blockDim.x) {
        double v = src[e];
        for (int p = 1; p < it.nparts; ++p) v += src[(long long)p * cnt + e]; /* fixed order: deterministic */
        dst[(long long)(e / it.tn) * it.ldc + (e % it.tn)] = v;
    }
}
void run_reduce(Stream* st, const ReduceItem* d_items, int nitems, double* y, const double* w) {
    if (nitems <= 0) return;
    reduce_kernel<<<nitems, 256, 0, st->s>>>(d_items, y, w);
    LAUNCH_CHECK();
}

/* ================================================================================================
 *  Lanczos vector kernels — HBM-bound streaming kernels, 16-byte vector loads where aligned,
 *  warp-shuffle + shared reductions, deterministic two-stage sums (no atomics).
 * ============================================================================================== */
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long z) {
    z += 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__global__ void fill_random_kernel(double* x, long long n, unsigned long long seed, long long first) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        x[i] = (double)(splitmix64(seed + (unsigned long long)(first + i) * 0x9E3779B97F4A7C15ULL) >> 11) / 9007199254740992.0 - 0.5;
}
void fill_random(Stream* st, double* x, long long n, unsigned long long seed, long long first) {
    if (n <= 0) return;
    int blocks = (int)std::min<long long>((n + 255) / 256, RED_BLOCKS);
    fill_random_kernel<<<blocks, 256, 0, st->s>>>(x, n, seed, first);
    LAUNCH_CHECK();
}

/* ---- fused Gram-Schmidt pass -------------------------------------------------------------------
 *  HBM-bound: one streaming read of nvec basis vectors (+ one read / optional write of w) per pass.  Each thread keeps
 *  its basis elements in registers between the update and the dot products, so the "reorthogonalise and measure" step
 *  costs one pass instead of two.  Block partial sums go to a scratch table; the block that draws the last ticket adds
 *  them in block order (a fixed order: bit-reproducible, no floating-point atomics). */
template <int NV>
__global__ void __launch_bounds__(256) gs_pass_kernel(const double* __restrict__ V, long long ldv, int nvec, double* __restrict__ w, long long n,
                                                      const double* __restrict__ coef, double* __restrict__ dots, double* __restrict__ nrm2,
                                                      double* __restrict__ partials, unsigned int* __restrict__ ticket) {
    __shared__ double c[NV];
    __shared__ double sh[NV + 1][8];
    __shared__ bool last;
    if (threadIdx.x < NV) c[threadIdx.x] = (coef && threadIdx.x < nvec) ? coef[threadIdx.x] : 0.0;
    __syncthreads();
    double s[NV + 1];
#pragma unroll
    for (int i = 0; i <= NV; ++i) s[i] = 0.0;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        double v[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) v[i] = i < nvec ? V[i * ldv + q] : 0.0;
        double wq = w[q];
        if (coef) {
#pragma unroll
            for (int i = 0; i < NV; ++i) wq -= c[i] * v[i];
            w[q] = wq;
        }
        if (dots) {
#pragma unroll
            for (int i = 0; i < NV; ++i) s[i] += v[i] * wq;
        }
        s[NV] += wq * wq;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i <= NV; ++i) {
        const double r = warp_sum(s[i]);
        if (lane == 0) sh[i][wid] = r;
    }
    __syncthreads();
    if (threadIdx.x <= NV) {
        double r = 0.0;
        for (int k = 0; k < 8; ++k) r += sh[threadIdx.x][k];
        partials[(long long)blockIdx.x * (NV + 1) + threadIdx.x] = r;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    /* the last block: warp `wid` sums columns wid, wid+8, ... over all blocks in block order */
    for (int i = wid; i <= NV; i += 8) {
        double r = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) r += partials[(long long)b * (NV + 1) + i];
        r = warp_sum(r);
        if (lane == 0) {
            if (i < NV) { if (dots && i < nvec) dots[i] = r; }
            else if (nrm2) *nrm2 = r;
        }
    }
    if (threadIdx.x == 0) *ticket = 0u;
}
void gs_pass(Stream* st, const double* V, long long ldv, int nvec, double* w, long long n, const double* d_coef, double* d_dots, double* d_nrm2) {
    if (nvec > RED_MAXVEC - 1) throw std::runtime_error("gs_pass: too many basis vectors");
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, RED_BLOCKS));
#define GS_LAUNCH(NV) gs_pass_kernel<NV><<<blocks, 256, 0, st->s>>>(V, ldv, nvec, w, n, d_coef, d_dots, d_nrm2, st->partials, st->ticket)
    if (nvec <= 4) GS_LAUNCH(4);
    else if (nvec <= 8) GS_LAUNCH(8);
    else if (nvec <= 12) GS_LAUNCH(12);
    else if (nvec <= 17) GS_LAUNCH(17);
    else if (nvec <= 24) GS_LAUNCH(24);
    else GS_LAUNCH(39);
#undef GS_LAUNCH
    LAUNCH_CHECK();
}
/* w = y is only read: gs_pass writes w only when it is given coefficients */
void dot(Stream* st, const double* x, const double* y, long long n, double* d_out) { gs_pass(st, x, n, 1, const_cast<double*>(y), n, nullptr, d_out, nullptr); }

/* ================================================================================================
 *  gram_kernel — G = PᵀP of a panel of np long columns (the correlation matrix, corr.cpp).  One CTA per (32×32 tile on or
 *  above the diagonal, slab of GR_SLAB rows).  Chunks of 64 rows of the tile's 32 + 32 columns are staged with 16-byte
 *  cp.async into a two-stage ring (a diagonal tile stages its columns once and reads them as both operands); warp w
 *  multiplies rows [16w, 16w+16) of every chunk into a full 32×32 DMMA accumulator (4×4 fragments), and the four warp
 *  partials are summed in shared memory in warp order.  The slab partial is written to a scratch area; gram_reduce_kernel
 *  sums the slabs in index order and writes both G[i][j] and G[j][i] from the same sum.  The columns are contiguous, so
 *  the arithmetic intensity is set by the tile width: about 4 flop per byte staged, ~np/4 per byte of DRAM traffic.
 *  RECT (gram_rect): G = PᵀQ of two panels, one CTA per (32×32 tile of every row tile of P × column tile of Q, slab), the same
 *  staging and DMMA body with no diagonal tile; gram_rect_reduce_kernel sums the slabs in index order into strided G.  An
 *  element's accumulator position, warp rows and slab order do not depend on np, nq or its tile, so its bits depend only on
 *  its two columns and n.
 * ============================================================================================== */
constexpr int GR_T = 32, GR_BK = 64, GR_S = GR_BK + 4 /* ≡ 4 mod 16: conflict-free fragment reads */, GR_THREADS = 128;
constexpr long long GR_SLAB = 8192;
constexpr int GR_STAGE = 2 * GR_T * GR_S; /* doubles of one stage: A and B columns */

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gsrc, int src_bytes) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gsrc), "r"(src_bytes));
}

/* symmetric (RECT false): Q = P, nt tiles per side, ntri tiles on or above the diagonal; RECT: nt = the tiles of Q, ntri = all tiles */
template <bool RECT>
__global__ void __launch_bounds__(GR_THREADS) gram_kernel(const double* __restrict__ P, long long ldp, int np, const double* __restrict__ Q, long long ldq,
                                                          int nq, long long n, int nt, int ntri, double* __restrict__ part) {
    extern __shared__ __align__(16) double gr_smem[];
    const int tri = blockIdx.x % ntri, slab = blockIdx.x / ntri;
    int ti = 0, tj = 0;
    if (RECT) { ti = tri / nt; tj = tri % nt; }
    else {
        int r = tri;
        while (r >= nt - ti) { r -= nt - ti; ++ti; }
        tj = ti + r;
    }
    const bool diag = !RECT && ti == tj;
    const long long r0 = (long long)slab * GR_SLAB, r1 = min(n, r0 + GR_SLAB);
    const int nchunks = (int)((r1 - r0 + GR_BK - 1) / GR_BK);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;

    /* this thread's eight 16-byte copies per operand: column q >> 5 of the tile, rows 2(q & 31), +1 of the chunk; columns past
       np are clamped to the last one (they only reach accumulator rows / columns that are never stored) */
    const double* srcA[8];
    const double* srcB[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int q = tid + GR_THREADS * i, col = q >> 5, pr = q & 31;
        srcA[i] = P + (long long)min(ti * GR_T + col, np - 1) * ldp + r0 + 2 * pr;
        srcB[i] = Q + (long long)min(tj * GR_T + col, nq - 1) * ldq + r0 + 2 * pr;
    }
    auto issue = [&](int c) {
        double* as = gr_smem + (c & 1) * GR_STAGE;
        double* bs = as + GR_T * GR_S;
        const long long row0 = r0 + (long long)c * GR_BK;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int q = tid + GR_THREADS * i, col = q >> 5, pr = q & 31;
            /* rows past the slab are zero-filled: a partial copy reads only the row that belongs to it */
            const long long left = r1 - (row0 + 2 * pr);
            const int bytes = left >= 2 ? 16 : (left == 1 ? 8 : 0);
            const long long adv = (long long)c * GR_BK;
            cp_async16(as + col * GR_S + 2 * pr, bytes ? srcA[i] + adv : P, bytes);
            if (!diag) cp_async16(bs + col * GR_S + 2 * pr, bytes ? srcB[i] + adv : Q, bytes);
        }
    };

    double acc[4][4][2];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }

    if (nchunks > 0) issue(0);
    cp_async_commit();
    for (int c = 0; c < nchunks; ++c) {
        if (c + 1 < nchunks) issue(c + 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        const double* as = gr_smem + (c & 1) * GR_STAGE;
        const double* bs = diag ? as : as + GR_T * GR_S;
        const int kb = warp * 16 + t;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            double a[4], b[4];
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) a[mi] = as[(mi * 8 + g) * GR_S + kb + 4 * kk];
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) b[ni] = bs[(ni * 8 + g) * GR_S + kb + 4 * kk];
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
        }
        __syncthreads();
    }
    cp_async_wait<0>();
    __syncthreads();
    /* the four warp partials, summed in warp order */
    double* red = gr_smem;
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
            double* p = red + warp * GR_T * GR_T + (mi * 8 + g) * GR_T + ni * 8 + 2 * t;
            p[0] = acc[mi][ni][0];
            p[1] = acc[mi][ni][1];
        }
    __syncthreads();
    double* out = part + ((long long)slab * ntri + tri) * (GR_T * GR_T);
    for (int e = tid; e < GR_T * GR_T; e += GR_THREADS)
        out[e] = ((red[e] + red[GR_T * GR_T + e]) + red[2 * GR_T * GR_T + e]) + red[3 * GR_T * GR_T + e];
}

__global__ void __launch_bounds__(256) gram_reduce_kernel(const double* __restrict__ part, int np, int nt, int ntri, int nslabs, double* __restrict__ G) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= (long long)np * np) return;
    int i = (int)(e / np), j = (int)(e % np);
    if (i > j) { const int s = i; i = j; j = s; }
    const int ti = i / GR_T, tj = j / GR_T;
    const int tri = ti * nt - ti * (ti - 1) / 2 + (tj - ti);
    const double* p = part + (long long)tri * (GR_T * GR_T) + (i % GR_T) * GR_T + (j % GR_T);
    double s = 0.0;
    for (int k = 0; k < nslabs; ++k) s += p[(long long)k * ntri * (GR_T * GR_T)];
    G[e] = s;
}

void gram(Stream* st, const double* P, long long ldp, int np, long long n, double* d_G) {
    if (np <= 0) return;
    if (n <= 0) { memset0(st, d_G, sizeof(double) * np * np); return; }
    if ((ldp & 1) || ((uintptr_t)P & 15)) throw std::runtime_error("gram: columns must be 16-byte aligned (P aligned, ldp even)");
    const int nt = (np + GR_T - 1) / GR_T, ntri = nt * (nt + 1) / 2;
    const long long nslabs = (n + GR_SLAB - 1) / GR_SLAB;
    constexpr int smem = 2 * GR_STAGE * (int)sizeof(double);
    static_assert(4 * GR_T * GR_T <= 2 * GR_STAGE, "the warp partials reuse the staging buffers");
    if (!st->gram_cfg) {
        CUDA_OK(cudaFuncSetAttribute(gram_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        st->gram_cfg = true;
    }
    double* part = (double*)malloc_bytes(st, sizeof(double) * nslabs * ntri * GR_T * GR_T);
    gram_kernel<false><<<(unsigned)(nslabs * ntri), GR_THREADS, smem, st->s>>>(P, ldp, np, P, ldp, np, n, nt, ntri, part);
    LAUNCH_CHECK();
    gram_reduce_kernel<<<(unsigned)(((long long)np * np + 255) / 256), 256, 0, st->s>>>(part, np, nt, ntri, (int)nslabs, d_G);
    LAUNCH_CHECK();
    free_bytes(st, part); /* stream-ordered heap: the next user of the range is queued behind the reduction */
}

__global__ void __launch_bounds__(256) gram_rect_reduce_kernel(const double* __restrict__ part, int np, int nq, int ntq, int ntiles, int nslabs,
                                                               double* __restrict__ G, long long gs, long long gc) {
    const long long e = (long long)blockIdx.x * 256 + threadIdx.x;
    if (e >= (long long)np * nq) return;
    const int i = (int)(e / nq), j = (int)(e % nq);
    const double* p = part + (long long)((i / GR_T) * ntq + j / GR_T) * (GR_T * GR_T) + (i % GR_T) * GR_T + (j % GR_T);
    double s = 0.0;
    for (int k = 0; k < nslabs; ++k) s += p[(long long)k * ntiles * (GR_T * GR_T)];
    G[i * gs + j * gc] = s;
}

void gram_rect(Stream* st, const double* P, long long ldp, int np, const double* Q, long long ldq, int nq, long long n, double* d_G, long long gs,
               long long gc) {
    if (np <= 0 || nq <= 0) return;
    if ((ldp & 1) || (ldq & 1) || ((uintptr_t)P & 15) || ((uintptr_t)Q & 15))
        throw std::runtime_error("gram_rect: columns must be 16-byte aligned (P and Q aligned, ldp and ldq even)");
    const int ntp = (np + GR_T - 1) / GR_T, ntq = (nq + GR_T - 1) / GR_T, ntiles = ntp * ntq;
    const long long nslabs = n > 0 ? (n + GR_SLAB - 1) / GR_SLAB : 0;
    constexpr int smem = 2 * GR_STAGE * (int)sizeof(double);
    double* part = nullptr;
    if (nslabs > 0) {
        if (!st->gram_rect_cfg) {
            CUDA_OK(cudaFuncSetAttribute(gram_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            st->gram_rect_cfg = true;
        }
        part = (double*)malloc_bytes(st, sizeof(double) * nslabs * ntiles * GR_T * GR_T);
        gram_kernel<true><<<(unsigned)(nslabs * ntiles), GR_THREADS, smem, st->s>>>(P, ldp, np, Q, ldq, nq, n, ntq, ntiles, part);
        LAUNCH_CHECK();
    }
    /* n <= 0: no slab, every element written as 0 */
    gram_rect_reduce_kernel<<<(unsigned)(((long long)np * nq + 255) / 256), 256, 0, st->s>>>(part, np, nq, ntq, ntiles, (int)nslabs, d_G, gs, gc);
    LAUNCH_CHECK();
    if (part) free_bytes(st, part);
}

/* ================================================================================================
 *  lanczos_kernel — one pass of the batched continued-fraction recurrence (spectral.cpp, dev.h: lanczos_batch).  CTA
 *  blockIdx.x = column · nblk + block: the column's rows are strided over its nblk blocks (nblk from n only), each block
 *  writes one partial, and the block that draws the column's last ticket adds the nblk partials in block order and updates
 *  that column's scalars.  HBM-bound streaming: pass 1 reads three vectors and writes two, pass 2 reads two and writes one.
 * ============================================================================================== */
constexpr int LZ_THREADS = 256;
int lanczos_blocks(long long n) { return (int)std::max<long long>(1, std::min<long long>((n + 4 * LZ_THREADS - 1) / (4 * LZ_THREADS), RED_BLOCKS)); }

__global__ void __launch_bounds__(LZ_THREADS) lanczos_kernel(LanczosBatch L, int pass, int t, int nblk, const double* __restrict__ prev,
                                                             double* __restrict__ cur, double* __restrict__ y) {
    const int col = blockIdx.x / nblk, blk = blockIdx.x % nblk;
    /* done is only written by the finisher of a column, after every block of that column has passed this test */
    if (L.done[col]) return;
    const long long off = (long long)col * L.ld, stride = (long long)nblk * LZ_THREADS;
    double* u = cur + off;
    double* w = y + off;
    double s = 0.0;
    if (pass == 0) {
        for (long long q = (long long)blk * LZ_THREADS + threadIdx.x; q < L.n; q += stride) { const double x = w[q]; s += x * x; }
    } else if (pass == 1) {
        const double c = L.scale[col], inv = 1.0 / c;
        if (t > 0) {
            const double* p = prev + off;
            for (long long q = (long long)blk * LZ_THREADS + threadIdx.x; q < L.n; q += stride) {
                const double v = u[q] * inv, x = w[q] * inv - c * p[q];
                u[q] = v; w[q] = x; s += v * x;
            }
        } else {
            for (long long q = (long long)blk * LZ_THREADS + threadIdx.x; q < L.n; q += stride) {
                const double v = u[q] * inv, x = w[q] * inv;
                u[q] = v; w[q] = x; s += v * x;
            }
        }
    } else {
        const double a = L.a[col];
        for (long long q = (long long)blk * LZ_THREADS + threadIdx.x; q < L.n; q += stride) { const double x = w[q] - a * u[q]; w[q] = x; s += x * x; }
    }
    __shared__ double sh[LZ_THREADS / 32];
    __shared__ bool last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    s = warp_sum(s);
    if (lane == 0) sh[wid] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
        for (int k = 0; k < LZ_THREADS / 32; ++k) r += sh[k];
        L.partials[(long long)col * nblk + blk] = r;
        __threadfence();
        last = atomicAdd(&L.tickets[col], 1u) == (unsigned)nblk - 1;
    }
    __syncthreads();
    if (!last || wid != 0) return;
    __threadfence();
    double r = 0.0;
    for (int b = lane; b < nblk; b += 32) r += __ldcg(L.partials + (long long)col * nblk + b);
    r = warp_sum(r);
    if (lane != 0) return;
    L.tickets[col] = 0u;
    if (pass == 0) {
        const bool zero = r <= L.zero2[col];
        L.norm2[col] = zero ? 0.0 : r;
        if (zero) L.done[col] = 1;
        else L.scale[col] = sqrt(r);
    } else if (pass == 1) {
        L.a[col] = r;
        L.alpha[(long long)col * L.nsteps + t] = r;
        if (t == L.nsteps - 1) { L.ndone[col] = L.nsteps; L.done[col] = 1; }
    } else {
        const double beta = sqrt(r), bt = t > 0 ? L.scale[col] : 0.0, a = L.a[col];
        if (beta <= LANCZOS_BETA_REL * sqrt(a * a + bt * bt)) { L.ndone[col] = t + 1; L.done[col] = 1; }
        else { L.beta[(long long)col * L.nsteps + t + 1] = beta; L.scale[col] = beta; }
    }
}

void lanczos_batch(Stream* st, const LanczosBatch& L, int pass, int t, const double* prev, double* cur, double* y) {
    if (L.nb <= 0 || L.n <= 0) return;
    const int nblk = lanczos_blocks(L.n);
    lanczos_kernel<<<(unsigned)((long long)L.nb * nblk), LZ_THREADS, 0, st->s>>>(L, pass, t, nblk, prev, cur, y);
    LAUNCH_CHECK();
}

template <int NV>
__global__ void __launch_bounds__(256) gs_final_kernel(const double* __restrict__ V, long long ldv, int nvec, const double* __restrict__ w, long long n,
                                                       const double* __restrict__ coef, const double* __restrict__ nrm2_in, double* __restrict__ nrm2_out,
                                                       double* __restrict__ vout) {
    __shared__ double c[NV];
    __shared__ double inv;
    __shared__ bool skip;
    if (threadIdx.x < NV) c[threadIdx.x] = threadIdx.x < nvec ? coef[threadIdx.x] : 0.0;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int i = 0; i < nvec; ++i) s += c[i] * c[i]; /* fixed order: every block (and every rank) gets the same bits */
        const double nin = *nrm2_in;
        /* refinement "if needed": a second-pass correction below GS_REFINE_REL of the vector's norm is not applied (the basis
           stays orthogonal to 1e-12, far inside what the Ritz values need); the pass is then one read and one write of w */
        const bool sk = s <= GS_REFINE_REL * GS_REFINE_REL * nin;
        double b2 = sk ? nin : nin - s;
        if (!(b2 > 0.0)) b2 = 0.0;
        inv = b2 > 0.0 ? 1.0 / sqrt(b2) : 0.0;
        skip = sk;
        if (blockIdx.x == 0) *nrm2_out = b2;
    }
    __syncthreads();
    const double sc = inv;
    if (skip) {
        for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) vout[q] = w[q] * sc;
        return;
    }
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        double v[NV]; /* every load is issued before the first use */
#pragma unroll
        for (int i = 0; i < NV; ++i) v[i] = i < nvec ? V[i * ldv + q] : 0.0;
        double acc = w[q];
#pragma unroll
        for (int i = 0; i < NV; ++i) acc -= c[i] * v[i];
        vout[q] = acc * sc;
    }
}
void gs_final(Stream* st, const double* V, long long ldv, int nvec, const double* w, long long n, const double* d_coef, const double* d_nrm2_in,
              double* d_nrm2_out, double* vout) {
    if (nvec > RED_MAXVEC) throw std::runtime_error("gs_final: too many basis vectors");
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, RED_BLOCKS));
#define GF_LAUNCH(NV) gs_final_kernel<NV><<<blocks, 256, 0, st->s>>>(V, ldv, nvec, w, n, d_coef, d_nrm2_in, d_nrm2_out, vout)
    if (nvec <= 4) GF_LAUNCH(4);
    else if (nvec <= 8) GF_LAUNCH(8);
    else if (nvec <= 12) GF_LAUNCH(12);
    else if (nvec <= 17) GF_LAUNCH(17);
    else if (nvec <= 24) GF_LAUNCH(24);
    else GF_LAUNCH(40);
#undef GF_LAUNCH
    LAUNCH_CHECK();
}

__global__ void scale_inv_norm_kernel(const double* __restrict__ w, const double* __restrict__ nrm2, double* __restrict__ v, long long n) {
    const double inv = 1.0 / sqrt(*nrm2);
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) v[q] = w[q] * inv;
}
void scale_inv_norm(Stream* st, const double* w, const double* d_nrm2, double* v, long long n) {
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, RED_BLOCKS));
    scale_inv_norm_kernel<<<blocks, 256, 0, st->s>>>(w, d_nrm2, v, n);
    LAUNCH_CHECK();
}

constexpr int RITZ_MAX = 40;
__global__ void __launch_bounds__(256) ritz_rotate_kernel(double* __restrict__ V, long long ldv, long long n, int ncv, const double* __restrict__ S,
                                                          int kk) {
    extern __shared__ double sS[]; /* ncv*kk */
    for (int i = threadIdx.x; i < ncv * kk; i += blockDim.x) sS[i] = S[i];
    __syncthreads();
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
        double v[RITZ_MAX];
#pragma unroll 8
        for (int i = 0; i < RITZ_MAX; ++i)
            if (i < ncv) v[i] = V[i * ldv + q];
        for (int a = 0; a < kk; ++a) {
            double o = 0.0;
            for (int i = 0; i < ncv; ++i) o += sS[i * kk + a] * v[i];
            V[a * ldv + q] = o;
        }
    }
}
void ritz_rotate(Stream* st, double* V, long long ldv, long long n, int ncv, const double* d_S, int kk) {
    if (ncv > RITZ_MAX) throw std::runtime_error("ritz_rotate: ncv too large");
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, RED_BLOCKS));
    ritz_rotate_kernel<<<blocks, 256, sizeof(double) * ncv * kk, st->s>>>(V, ldv, n, ncv, d_S, kk);
    LAUNCH_CHECK();
}

__global__ void filter_small_kernel(double* x, long long n, double tol) {
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x)
        if (fabs(x[q]) < tol) x[q] = 0.0;
}
void filter_small(Stream* st, double* x, long long n, double tol) {
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, RED_BLOCKS));
    filter_small_kernel<<<blocks, 256, 0, st->s>>>(x, n, tol);
    LAUNCH_CHECK();
}

__global__ void axpby_out_kernel(const double* a, const double* b, double alpha, double* out, long long n) {
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x)
        out[q] = (a ? a[q] : 0.0) + alpha * b[q];
}
void axpby_out(Stream* st, const double* a, const double* b, double alpha, double* out, long long n) {
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, RED_BLOCKS));
    axpby_out_kernel<<<blocks, 256, 0, st->s>>>(a, b, alpha, out, n);
    LAUNCH_CHECK();
}

__global__ void gather_rows_reversed_kernel(const double* __restrict__ src, int n, int m, double* __restrict__ dst) {
    const long long total = (long long)m * n;
    for (long long q = blockIdx.x * (long long)blockDim.x + threadIdx.x; q < total; q += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(q / n), i = (int)(q % n);
        dst[q] = src[(long long)(n - 1 - k) * n + i];
    }
}
void gather_rows_reversed(Stream* st, const double* src, int n, int m, double* dst) {
    if (m <= 0) return;
    const long long total = (long long)m * n;
    const int blocks = (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, RED_BLOCKS));
    gather_rows_reversed_kernel<<<blocks, 256, 0, st->s>>>(src, n, m, dst);
    LAUNCH_CHECK();
}

/* ================================================================================================
 *  Collectives: NCCL, bound lazily (dlopen) so that a single-GPU process never needs the library.  In a Python
 *  process torch has already loaded its bundled libnccl.so.2 and dlopen returns that same copy.
 * ============================================================================================== */
namespace {
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi& nccl() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api;
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { g_err = std::string("cannot load NCCL: ") + dlerror(); return api; }
#define BIND(name) api.name = (decltype(api.name))dlsym(h, "nccl" #name); if (!api.name) { g_err = "NCCL symbol nccl" #name " missing"; return api; }
    BIND(GetUniqueId) BIND(CommInitRank) BIND(CommDestroy) BIND(AllReduce) BIND(Broadcast) BIND(Send) BIND(Recv) BIND(GroupStart) BIND(GroupEnd) BIND(GetErrorString)
#undef BIND
    api.ok = true;
    return api;
}
}  // namespace
#define NCCL_OK(call)                                                                                     \
    do {                                                                                                  \
        ncclResult_t r_ = (call);                                                                         \
        if (r_ != ncclSuccess) {                                                                          \
            char buf_[512];                                                                               \
            snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, nccl().GetErrorString(r_)); \
            g_err = buf_;                                                                                 \
            fprintf(stderr, "[dmrgx] %s\n", buf_);                                                        \
            throw std::runtime_error(buf_);                                                               \
        }                                                                                                 \
    } while (0)

static void comm_destroy_(Stream* st) { if (st->comm && nccl().ok) nccl().CommDestroy(st->comm); st->comm = nullptr; }
int comm_unique_id(void* out) {
    static_assert(sizeof(ncclUniqueId) == COMM_ID_BYTES, "ncclUniqueId size");
    if (!nccl().ok) return 110;
    ncclUniqueId id;
    if (nccl().GetUniqueId(&id) != ncclSuccess) { g_err = "ncclGetUniqueId failed"; return 111; }
    std::memcpy(out, &id, sizeof id);
    return 0;
}
int comm_init(Stream* st, int rank, int world, const void* idbytes) {
    if (world <= 1) { st->rank = 0; st->world = 1; return 0; }
    if (!nccl().ok) return 110;
    ncclUniqueId id;
    std::memcpy(&id, idbytes, sizeof id);
    cudaSetDevice(st->device);
    ncclResult_t r = nccl().CommInitRank(&st->comm, world, id, rank);
    if (r != ncclSuccess) { g_err = std::string("ncclCommInitRank failed: ") + nccl().GetErrorString(r); return 112; }
    st->rank = rank; st->world = world;
    return 0;
}
void allreduce_sum(Stream* st, double* d_buf, long long n) {
    if (st->world <= 1 || n <= 0) return;
    NCCL_OK(nccl().AllReduce(d_buf, d_buf, (size_t)n, ncclDouble, ncclSum, st->comm, st->s));
}
/* Ragged in-place all-gather as ONE group of point-to-point transfers: every rank sends its own range to each peer and
   receives each peer's range straight into place.  Through NVSwitch all pairs run at full bandwidth at once, and the
   group is a single NCCL kernel — a chain of per-root broadcasts cost 0.1-0.3 ms at 4-8 ranks for 15 MB. */
void allgatherv(Stream* st, double* d_buf, const long long* off) {
    if (st->world <= 1) return;
    const long long mine = off[st->rank + 1] - off[st->rank];
    NCCL_OK(nccl().GroupStart());
    for (int d = 1; d < st->world; ++d) {
        const int to = (st->rank + d) % st->world, from = (st->rank - d + st->world) % st->world;
        if (mine > 0) NCCL_OK(nccl().Send(d_buf + off[st->rank], (size_t)mine, ncclDouble, to, st->comm, st->s));
        const long long cnt = off[from + 1] - off[from];
        if (cnt > 0) NCCL_OK(nccl().Recv(d_buf + off[from], (size_t)cnt, ncclDouble, from, st->comm, st->s));
    }
    NCCL_OK(nccl().GroupEnd());
}
void exchange_ranges(Stream* st, double* d_buf, int n, const int* from, const int* to, const long long* off, const long long* cnt) {
    if (st->world <= 1 || n <= 0) return;
    NCCL_OK(nccl().GroupStart());
    for (int i = 0; i < n; ++i) {
        if (cnt[i] <= 0 || from[i] == to[i]) continue;
        if (from[i] == st->rank) NCCL_OK(nccl().Send(d_buf + off[i], (size_t)cnt[i], ncclDouble, to[i], st->comm, st->s));
        if (to[i] == st->rank) NCCL_OK(nccl().Recv(d_buf + off[i], (size_t)cnt[i], ncclDouble, from[i], st->comm, st->s));
    }
    NCCL_OK(nccl().GroupEnd());
}
void bcast_batch(Stream* st, int n, double* const* d_ptr, const long long* count, const int* root) {
    if (st->world <= 1 || n <= 0) return;
    NCCL_OK(nccl().GroupStart());
    for (int i = 0; i < n; ++i)
        if (count[i] > 0) NCCL_OK(nccl().Broadcast(d_ptr[i], d_ptr[i], (size_t)count[i], ncclDouble, root[i], st->comm, st->s));
    NCCL_OK(nccl().GroupEnd());
}

/* ================================================================================================
 *  Small reduced-density-matrix blocks (n <= 64): batched cyclic Jacobi, one CTA per block, the block and its
 *  eigenvector matrix in shared memory.  A round of the round-robin schedule holds n/2 disjoint index pairs; their
 *  rotations are computed from the current matrix and applied together (columns, then rows), so a sweep is n-1 rounds
 *  of fully parallel updates.  Jacobi is accurate to working precision in the small eigenvalues too, which is what the
 *  truncation ranks.  Larger blocks go to the block-Jacobi kernels below.
 *  Replaces EigRDM_BlockDiag / EPSLAPACK (include/DMRGBlockContainer.hpp:1962-2003) for these sizes.
 * ============================================================================================== */
constexpr int JAC_NMAX = 64, JAC_LD = JAC_NMAX + 1, JAC_THREADS = 256;
struct JacobiJob { double* A; double* w; int n; int pad; };

__global__ void __launch_bounds__(JAC_THREADS) jacobi_eig_kernel(const JacobiJob* __restrict__ jobs) {
    extern __shared__ double jsm[];
    double* A = jsm;                       /* [JAC_NMAX][JAC_LD] */
    double* V = jsm + JAC_NMAX * JAC_LD;   /* eigenvectors in columns */
    __shared__ double cs[JAC_NMAX / 2][2];
    __shared__ int pq[JAC_NMAX / 2][2];
    __shared__ double red[JAC_THREADS / 32][2];
    __shared__ double offdiag[2];
    const JacobiJob job = jobs[blockIdx.x];
    const int n = job.n, tid = threadIdx.x;
    const int ne = (n + 1) & ~1; /* the schedule needs an even count: an odd block gets an idle dummy index */
    for (int e = tid; e < n * n; e += JAC_THREADS) {
        const int i = e / n, j = e % n;
        A[i * JAC_LD + j] = job.A[e];
        V[i * JAC_LD + j] = i == j ? 1.0 : 0.0;
    }
    __syncthreads();
    for (int sweep = 0; sweep < 40; ++sweep) {
        /* convergence: off-diagonal weight against the diagonal's */
        double off = 0.0, dg = 0.0;
        for (int e = tid; e < n * n; e += JAC_THREADS) {
            const int i = e / n, j = e % n;
            const double a = A[i * JAC_LD + j];
            if (i == j) dg += a * a; else off += a * a;
        }
        off = warp_sum(off); dg = warp_sum(dg);
        if ((tid & 31) == 0) { red[tid >> 5][0] = off; red[tid >> 5][1] = dg; }
        __syncthreads();
        if (tid == 0) {
            double o = 0, d = 0;
            for (int k = 0; k < JAC_THREADS / 32; ++k) { o += red[k][0]; d += red[k][1]; }
            offdiag[0] = o; offdiag[1] = d;
        }
        __syncthreads();
        if (offdiag[0] == 0.0 || offdiag[0] <= 1e-33 * (offdiag[0] + offdiag[1])) break;
        for (int round = 0; round < ne - 1; ++round) {
            /* round-robin pairing: index ne-1 stays, the others rotate */
            if (tid < ne / 2) {
                int a = tid == 0 ? ne - 1 : (round + tid) % (ne - 1);
                int b = (round + ne - 1 - tid) % (ne - 1);
                int p = a < b ? a : b, q = a < b ? b : a;
                double c = 1.0, sn = 0.0;
                if (q < n) {
                    const double apq = A[p * JAC_LD + q];
                    if (apq != 0.0) {
                        const double theta = (A[q * JAC_LD + q] - A[p * JAC_LD + p]) / (2.0 * apq);
                        const double tt = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                        c = 1.0 / sqrt(tt * tt + 1.0);
                        sn = tt * c;
                    }
                } else { p = -1; }
                pq[tid][0] = p; pq[tid][1] = q;
                cs[tid][0] = c; cs[tid][1] = sn;
            }
            __syncthreads();
            /* columns p,q of A and of V */
            for (int e = tid; e < (ne / 2) * n; e += JAC_THREADS) {
                const int k = e / n, i = e % n;
                const int p = pq[k][0], q = pq[k][1];
                if (p < 0) continue;
                const double c = cs[k][0], sn = cs[k][1];
                const double x = A[i * JAC_LD + p], y = A[i * JAC_LD + q];
                A[i * JAC_LD + p] = c * x - sn * y; A[i * JAC_LD + q] = sn * x + c * y;
                const double vx = V[i * JAC_LD + p], vy = V[i * JAC_LD + q];
                V[i * JAC_LD + p] = c * vx - sn * vy; V[i * JAC_LD + q] = sn * vx + c * vy;
            }
            __syncthreads();
            /* rows p,q of A */
            for (int e = tid; e < (ne / 2) * n; e += JAC_THREADS) {
                const int k = e / n, j = e % n;
                const int p = pq[k][0], q = pq[k][1];
                if (p < 0) continue;
                const double c = cs[k][0], sn = cs[k][1];
                const double x = A[p * JAC_LD + j], y = A[q * JAC_LD + j];
                A[p * JAC_LD + j] = c * x - sn * y; A[q * JAC_LD + j] = sn * x + c * y;
            }
            __syncthreads();
        }
    }
    /* ascending order by rank (stable on ties); row k of the output = k-th eigenvector */
    __shared__ int rank_of[JAC_NMAX];
    if (tid < n) {
        const double di = A[tid * JAC_LD + tid];
        int r = 0;
        for (int j = 0; j < n; ++j) { const double dj = A[j * JAC_LD + j]; r += (dj < di || (dj == di && j < tid)) ? 1 : 0; }
        rank_of[tid] = r;
        job.w[r] = di;
    }
    __syncthreads();
    for (int e = tid; e < n * n; e += JAC_THREADS) {
        const int col = e / n, i = e % n; /* eigenvector `col` of V, component i */
        job.A[(long long)rank_of[col] * n + i] = V[i * JAC_LD + col];
    }
}

/* ================================================================================================
 *  Reduced-density-matrix blocks above 64 states: batched two-sided BLOCK Jacobi, all blocks of both sides in the same
 *  launches, no host threads, no vendor library (replaces EigRDM_BlockDiag / EPSLAPACK, include/DMRGBlockContainer.hpp:
 *  1962-2003, for every size).  A matrix is padded to a multiple of 64 and cut into 32-wide blocks; a round of the
 *  round-robin tournament pairs the blocks (I_k, J_k), k < nb/2:
 *    eig_sub_kernel    one CTA per pair: the 64x64 symmetric sub-problem [[A_II, A_IJ], [A_JI, A_JJ]] is gathered into shared
 *                      memory and diagonalised by parallel-ordered cyclic Jacobi (all angles <= pi/4, so the rotation Q_k stays
 *                      the orthogonal matrix nearest the identity: no eigenvalue swaps, which is what makes the outer
 *                      iteration converge); writes Q_k and the diagonalised sub-problem back;
 *    eig_apply_kernel  FP64 DMMA: one CTA per 64x64 tile A[(I_k,J_k),(I_k',J_k')] <- Q_k^T · tile · Q_k' (k < k', the mirror
 *                      tile is written as the transpose: A stays exactly symmetric) and per 64-column chunk of the eigenvector
 *                      rows VT[(I_k,J_k), :] <- Q_k^T · VT[(I_k,J_k), :]; tiles whose pairs did not rotate are skipped.
 *  A sweep is nb-1 rounds; sub-problems whose off-diagonal weight is below 1e-34 of the matrix' squared Frobenius norm do
 *  not rotate, and a matrix is finished after a sweep without rotation (the host reads one flag per matrix per sweep of
 *  the largest matrix).  Jacobi's accuracy in the small eigenvalues is what the truncation ranks.
 * ============================================================================================== */
constexpr int EB = 32;               /* block width */
constexpr int ET = 2 * EB;           /* sub-problem / tile extent */
constexpr int ELD = ET + 4;          /* shared-memory row stride (68 = 4 mod 16 doubles: conflict-free fragment reads both ways) */
struct EigJob {
    double* A;       /* np x np, row-major, padded with zeros */
    double* VT;      /* np x np: row i = current i-th eigenvector estimate */
    double* Q;       /* (nb/2) x 64 x 64 rotations of the current round */
    int* rot;        /* (nb/2): the pair rotated in the current round */
    double* outA;    /* n x n: row k = k-th eigenvector, ascending eigenvalues */
    double* outW;    /* n */
    double* norm2;   /* squared Frobenius norm */
    int* active;     /* any rotation since the flag was last cleared */
    int n, np, nb, pad;
};

/* round r of the round-robin tournament over nb (even) players: pair k = (a, b), a < b */
__device__ __forceinline__ void eig_pair(int nb, int r, int k, int& I, int& J) {
    const int a = k == 0 ? nb - 1 : (r + k) % (nb - 1);
    const int b = (r + nb - 1 - k) % (nb - 1);
    I = a < b ? a : b; J = a < b ? b : a;
}

/* Starting order: the coordinates sorted by DESCENDING diagonal entry.  In a DMRG step the basis of a block is (kept states of
   the previous step, already ordered by weight) x (site states), so the diagonal of rho is informative and the sorted matrix
   starts out graded — the form on which the sorted block Jacobi converges fastest.  perm[i] = original coordinate at position i
   (the rank array of the finish step doubles as scratch for it). */
__global__ void __launch_bounds__(256) eig_perm_kernel(const EigJob* __restrict__ jobs, int* __restrict__ perm_ws, const int* __restrict__ perm_off) {
    const EigJob jb = jobs[blockIdx.y];
    int* perm = perm_ws + perm_off[blockIdx.y];
    const int n = jb.n;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const double di = jb.outA[(long long)i * n + i];
        int rk = 0;
        for (int j = 0; j < n; ++j) { const double dj = jb.outA[(long long)j * n + j]; rk += (dj > di || (dj == di && j < i)) ? 1 : 0; }
        perm[rk] = i;
    }
}
__global__ void __launch_bounds__(256) eig_init_kernel(const EigJob* __restrict__ jobs, const int* __restrict__ perm_ws, const int* __restrict__ perm_off) {
    const EigJob jb = jobs[blockIdx.y];
    const int* perm = perm_ws + perm_off[blockIdx.y];
    const long long tot = (long long)jb.np * jb.np;
    for (long long e = blockIdx.x * 256ll + threadIdx.x; e < tot; e += (long long)gridDim.x * 256) {
        const int i = (int)(e / jb.np), j = (int)(e % jb.np);
        const bool in = i < jb.n && j < jb.n;
        jb.A[e] = in ? jb.outA[(long long)perm[i] * jb.n + perm[j]] : 0.0;
        jb.VT[e] = (i < jb.n ? perm[i] == j : i == j) ? 1.0 : 0.0; /* row i = unit vector of the original coordinate perm[i] */
    }
}
/* squared Frobenius norm, one CTA per matrix, fixed summation order (deterministic thresholds) */
__global__ void __launch_bounds__(1024) eig_norm_kernel(const EigJob* __restrict__ jobs) {
    const EigJob jb = jobs[blockIdx.x];
    __shared__ double red[32];
    double s = 0.0;
    const long long tot = (long long)jb.n * jb.n;
    for (long long e = threadIdx.x; e < tot; e += 1024) { const double v = jb.outA[e]; s += v * v; }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = warp_sum(red[threadIdx.x]);
        if (threadIdx.x == 0) { *jb.norm2 = s; *jb.active = 0; }
    }
}

/* job and local index of a CTA from the prefix table (njobs+1 entries) */
__device__ __forceinline__ int eig_find(const int* __restrict__ prefix, int njobs, int cta, int& local) {
    int lo = 0, hi = njobs;
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (prefix[mid] <= cta) lo = mid; else hi = mid; }
    local = cta - prefix[lo];
    return lo;
}

constexpr int ESUB_THREADS = 1024; /* the sub-problem is latency-bound (three barriers per rotation round): all the threads an SM has */
/* one CTA per SM, stated: with it the compiler spends the 64 registers a thread has on keeping the rotation rounds'
   thread-invariant shared-memory addresses instead of recomputing them from threadIdx every round (without it: 48
   registers, and tools/eig_probe.py 2048 solves 5 % slower on a B200 at 1000 W) */
__global__ void __launch_bounds__(ESUB_THREADS, 1) eig_sub_kernel(const EigJob* __restrict__ jobs, const int* __restrict__ prefix, int njobs, int round, bool first) {
    extern __shared__ double jsm[];
    double* A = jsm;                 /* [64][65] */
    double* V = jsm + ET * JAC_LD;   /* rotation, columns = eigenvectors */
    __shared__ double cs[ET / 2][2];
    __shared__ int pq[ET / 2][2];
    __shared__ double red[ESUB_THREADS / 32], redw[ESUB_THREADS / 32];
    __shared__ double offsh, offwsh;
    int k;
    const EigJob jb = jobs[eig_find(prefix, njobs, blockIdx.x, k)];
    const int tid = threadIdx.x, np = jb.np;
    int I, J;
    eig_pair(jb.nb, round % (jb.nb - 1), k, I, J);
    for (int e = tid; e < ET * ET; e += ESUB_THREADS) {
        const int i = e >> 6, j = e & 63;
        const int gi = (i < EB ? I * EB + i : J * EB + i - EB), gj = (j < EB ? I * EB + j : J * EB + j - EB);
        A[i * JAC_LD + j] = jb.A[(long long)gi * np + gj];
        V[i * JAC_LD + j] = i == j ? 1.0 : 0.0;
    }
    __syncthreads();
    /* A sub-problem rotates while its off-diagonal weight exceeds the noise the FP64 DMMA updates leave in it (about
       sqrt(64)·eps of the matrix norm per element and round): off(S) <= 3e-14·||A||_F.  The eigenvalues are afterwards taken as
       Rayleigh quotients with the original matrix, which squares this error. */
    const double thr = 1e-27 * *jb.norm2;
    bool rotated = false;
    for (int sweep = 0; sweep < 2; ++sweep) {
        double off = 0.0, offw = 0.0; /* off-diagonal weight: all of it / the part inside the two diagonal blocks */
        for (int e = tid; e < ET * ET; e += ESUB_THREADS) {
            const int i = e >> 6, j = e & 63;
            const double a = A[i * JAC_LD + j];
            if (i != j) { off += a * a; if ((i < EB) == (j < EB)) offw += a * a; }
        }
        off = warp_sum(off); offw = warp_sum(offw);
        if ((tid & 31) == 0) { red[tid >> 5] = off; redw[tid >> 5] = offw; }
        __syncthreads();
        if (tid == 0) { double o = 0, ow = 0; for (int w = 0; w < ESUB_THREADS / 32; ++w) { o += red[w]; ow += redw[w]; } offsh = o; offwsh = ow; }
        __syncthreads();
        if (offsh <= thr) break;
        rotated = true;
        /* two inner sweeps: FULL cyclic sweeps (63 rounds: all 2016 pairs) in the first outer sweep of the solve; after it a
           CROSS sweep (32 rounds: the 1024 pairs (p in block I, q in block J) only — where the off-diagonal weight sits once
           both diagonal blocks have been diagonalised by an earlier visit), then a full one.  A sweep that finds no weight
           left inside the two diagonal blocks is a cross sweep. */
        const bool full = (first || sweep == 1) && offwsh > 0.0;
        const int nrounds = full ? ET - 1 : EB;
        for (int rr = 0; rr < nrounds; ++rr) {
            if (tid < ET / 2) {
                int p, q;
                if (full) {
                    const int a = tid == 0 ? ET - 1 : (rr + tid) % (ET - 1);
                    const int b = (rr + ET - 1 - tid) % (ET - 1);
                    p = a < b ? a : b; q = a < b ? b : a;
                } else { p = tid; q = EB + ((tid + rr) & (EB - 1)); }
                double c = 1.0, sn = 0.0;
                const double apq = A[p * JAC_LD + q];
                /* the rotation with |angle| <= pi/4 that zeroes a_pq, with TWO dependent reciprocal square roots and no division
                   (this step is serial: every special function is latency on the critical path of the whole solver):
                   d = a_qq - a_pp, b = 2 a_pq, h = hypot(d, b):  c^2 = (h + |d|) / 2h,  c = c^2 / sqrt(c^2),  s = sgn(d) b / (2 h c);
                   c^2 + s^2 = 1 holds to round-off by construction */
                const double d = A[q * JAC_LD + q] - A[p * JAC_LD + p], b2 = 2.0 * apq;
                const double hh = d * d + b2 * b2;
                if (apq != 0.0 && hh > 1e-290) {
                    const double rh = rsqrt(hh);
                    const double c2 = 0.5 + 0.5 * fabs(d) * rh;
                    const double rc = rsqrt(c2);
                    c = c2 * rc;
                    sn = (d >= 0.0 ? 0.5 : -0.5) * b2 * rh * rc;
                }
                pq[tid][0] = p; pq[tid][1] = q;
                cs[tid][0] = c; cs[tid][1] = sn;
            }
            __syncthreads();
            /* A <- J^T A J and V <- V J in ONE phase: the 2x2 block {p1,q1} x {p2,q2} of A transforms on its own (one thread per
               block, 32 x 32 blocks), and so does every row of the column pair {p,q} of V — two barriers per round, not three */
            {
                const int k1 = tid >> 5, k2 = tid & 31;
                const int p1 = pq[k1][0], q1 = pq[k1][1], p2 = pq[k2][0], q2 = pq[k2][1];
                const double c1 = cs[k1][0], s1 = cs[k1][1], c2 = cs[k2][0], s2 = cs[k2][1];
                const double a11 = A[p1 * JAC_LD + p2], a12 = A[p1 * JAC_LD + q2], a21 = A[q1 * JAC_LD + p2], a22 = A[q1 * JAC_LD + q2];
                /* columns: [x y] <- [c x - s y, s x + c y] */
                const double b11 = c2 * a11 - s2 * a12, b12 = s2 * a11 + c2 * a12;
                const double b21 = c2 * a21 - s2 * a22, b22 = s2 * a21 + c2 * a22;
                /* rows: same with (c1, s1) */
                A[p1 * JAC_LD + p2] = c1 * b11 - s1 * b21; A[q1 * JAC_LD + p2] = s1 * b11 + c1 * b21;
                A[p1 * JAC_LD + q2] = c1 * b12 - s1 * b22; A[q1 * JAC_LD + q2] = s1 * b12 + c1 * b22;
#pragma unroll
                for (int e = tid; e < (ET / 2) * ET; e += ESUB_THREADS) {
                    const int kk = e >> 6, i = e & 63;
                    const int p = pq[kk][0], q = pq[kk][1];
                    const double c = cs[kk][0], sn = cs[kk][1];
                    const double vx = V[i * JAC_LD + p], vy = V[i * JAC_LD + q];
                    V[i * JAC_LD + p] = c * vx - sn * vy; V[i * JAC_LD + q] = sn * vx + c * vy;
                }
            }
            __syncthreads();
        }
    }
    /* The 64 diagonal entries are put in DESCENDING order (a permutation folded into Q): over a sweep the large eigenvalues
       migrate to the leading blocks, the matrix becomes graded along its diagonal and the small trailing part decouples —
       reduced density matrices have exponentially decaying spectra with tiny absolute gaps, and without the sorting the
       iteration spends ~25 sweeps in its linear phase (measured, profiles/r2_eigensolver.md). */
    __shared__ int rank_of[ET];
    __shared__ int moved;
    if (tid == 0) moved = 0;
    __syncthreads();
    if (tid < ET) {
        /* padding coordinates (global index >= n: exact zero rows / columns, never rotated) keep their trailing positions: a
           slightly negative round-off eigenvalue must not change places with them */
        const int gt = tid < EB ? I * EB + tid : J * EB + tid - EB;
        const bool pad_t = gt >= jb.n;
        const double di = A[tid * JAC_LD + tid];
        int rk = 0;
        for (int j = 0; j < ET; ++j) {
            const int gj = j < EB ? I * EB + j : J * EB + j - EB;
            const bool pad_j = gj >= jb.n;
            const double dj = A[j * JAC_LD + j];
            const bool before = pad_t != pad_j ? !pad_j : (dj > di || (dj == di && j < tid));
            rk += before ? 1 : 0;
        }
        rank_of[tid] = rk;
        if (rk != tid) moved = 1;
    }
    __syncthreads();
    const bool changed = rotated || moved;
    if (tid == 0) { jb.rot[k] = changed ? 1 : 0; if (rotated) *jb.active = 1; }
    if (!changed) return;
    double* Q = jb.Q + (long long)k * ET * ET;
    for (int e = tid; e < ET * ET; e += ESUB_THREADS) {
        const int i = e >> 6, j = e & 63;
        const int ri = rank_of[i], rj = rank_of[j];
        Q[i * ET + rj] = V[i * JAC_LD + j];
        /* the rotated sub-problem goes back in place (symmetrised: the two triangles differ by round-off) */
        const int gi = (ri < EB ? I * EB + ri : J * EB + ri - EB), gj = (rj < EB ? I * EB + rj : J * EB + rj - EB);
        jb.A[(long long)gi * np + gj] = i == j ? A[i * JAC_LD + j] : 0.5 * (A[i * JAC_LD + j] + A[j * JAC_LD + i]);
    }
}

/* 64x64x64 product from shared memory on the FP64 tensor pipe: acc = op(X) · Y with X(m,k) = xs[m*sxm + k*sxk], Y(k,n) = ys[k*ELD + n] */
__device__ __forceinline__ void eig_mma64(double (&acc)[4][4][2], const double* xs, int sxm, int sxk, const double* ys, int rbase, int cbase, int g, int t) {
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }
#pragma unroll 4
    for (int k0 = 0; k0 < ET; k0 += 4) {
        double a[4], b[4];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) a[mi] = xs[(rbase + mi * 8 + g) * sxm + (k0 + t) * sxk];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) b[ni] = ys[(k0 + t) * ELD + cbase + ni * 8 + g];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) dmma_m8n8k4(acc[mi][ni][0], acc[mi][ni][1], a[mi], b[ni]);
    }
}
__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gsrc) {
    unsigned sdst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sdst), "l"(gsrc));
}
/* rows (I-block, J-block) x 64 columns starting at the two 32-column pieces c0, c1 of a row-major np-wide matrix -> smem [64][ELD] */
__device__ __forceinline__ void eig_load_tile(double* dst, const double* M, int np, int I, int J, int c0, int c1, int tid) {
    for (int e = tid; e < ET * (ET / 2); e += 128) { /* 16-byte pieces */
        const int i = e >> 5, j2 = (e & 31) * 2;
        const int gi = (i < EB ? I * EB + i : J * EB + i - EB);
        const int gj = (j2 < EB ? c0 + j2 : c1 + j2 - EB);
        cp_async16(dst + i * ELD + j2, M + (long long)gi * np + gj);
    }
}

__global__ void __launch_bounds__(128, 2) eig_apply_kernel(const EigJob* __restrict__ jobs, const int* __restrict__ prefix, int njobs, int round) {
    extern __shared__ double esm[];
    double* T0 = esm;                 /* the tile, then the intermediate */
    double* Q0 = esm + ET * ELD;      /* Q_k  */
    double* Q1 = esm + 2 * ET * ELD;  /* Q_k' */
    int local;
    const EigJob jb = jobs[eig_find(prefix, njobs, blockIdx.x, local)];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const int rbase = (warp >> 1) * 32, cbase = (warp & 1) * 32;
    const int np = jb.np, npair = jb.nb / 2, r = round % (jb.nb - 1);
    const int ntri = npair * (npair - 1) / 2;
    double acc[4][4][2];
    if (local < ntri) {
        /* ---- A tile (k < k'): T = Q_k^T · A[(I,J),(I',J')] · Q_k' ---- */
        int k = 0, rem = local;
        while (rem >= npair - 1 - k) { rem -= npair - 1 - k; ++k; }
        const int k2 = k + 1 + rem;
        const int rk = jb.rot[k], rk2 = jb.rot[k2];
        if (!rk && !rk2) return;
        int I, J, I2, J2;
        eig_pair(jb.nb, r, k, I, J);
        eig_pair(jb.nb, r, k2, I2, J2);
        eig_load_tile(T0, jb.A, np, I, J, I2 * EB, J2 * EB, tid);
        if (rk) for (int e = tid; e < ET * (ET / 2); e += 128) cp_async16(Q0 + (e >> 5) * ELD + (e & 31) * 2, jb.Q + (long long)k * ET * ET + (e >> 5) * ET + (e & 31) * 2);
        if (rk2) for (int e = tid; e < ET * (ET / 2); e += 128) cp_async16(Q1 + (e >> 5) * ELD + (e & 31) * 2, jb.Q + (long long)k2 * ET * ET + (e >> 5) * ET + (e & 31) * 2);
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        if (rk2) { /* T0 <- T0 · Q_k' */
            eig_mma64(acc, T0, ELD, 1, Q1, rbase, cbase, g, t);
            __syncthreads();
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) {
                    double* p = T0 + (rbase + mi * 8 + g) * ELD + cbase + ni * 8 + 2 * t;
                    p[0] = acc[mi][ni][0]; p[1] = acc[mi][ni][1];
                }
            __syncthreads();
        }
        if (rk) eig_mma64(acc, Q0, 1, ELD, T0, rbase, cbase, g, t); /* Q_k^T · T0 */
        else {
#pragma unroll
            for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) {
                    const double* p = T0 + (rbase + mi * 8 + g) * ELD + cbase + ni * 8 + 2 * t;
                    acc[mi][ni][0] = p[0]; acc[mi][ni][1] = p[1];
                }
        }
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int i = rbase + mi * 8 + g, j = cbase + ni * 8 + 2 * t + hh;
                    const int gi = (i < EB ? I * EB + i : J * EB + i - EB), gj = (j < EB ? I2 * EB + j : J2 * EB + j - EB);
                    jb.A[(long long)gi * np + gj] = acc[mi][ni][hh];
                    jb.A[(long long)gj * np + gi] = acc[mi][ni][hh]; /* the mirror tile */
                }
    } else {
        /* ---- eigenvector rows: VT[(I,J), chunk] <- Q_k^T · VT[(I,J), chunk] ---- */
        const int nchunk = np / ET;
        const int k = (local - ntri) / nchunk, ch = (local - ntri) % nchunk;
        if (!jb.rot[k]) return;
        int I, J;
        eig_pair(jb.nb, r, k, I, J);
        eig_load_tile(T0, jb.VT, np, I, J, ch * ET, ch * ET + EB, tid);
        for (int e = tid; e < ET * (ET / 2); e += 128) cp_async16(Q0 + (e >> 5) * ELD + (e & 31) * 2, jb.Q + (long long)k * ET * ET + (e >> 5) * ET + (e & 31) * 2);
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        eig_mma64(acc, Q0, 1, ELD, T0, rbase, cbase, g, t);
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) {
                const int i = rbase + mi * 8 + g, j = cbase + ni * 8 + 2 * t;
                const int gi = (i < EB ? I * EB + i : J * EB + i - EB);
                double* p = jb.VT + (long long)gi * np + ch * ET + j;
                p[0] = acc[mi][ni][0]; p[1] = acc[mi][ni][1];
            }
    }
}

/* Eigenvalues as Rayleigh quotients with the ORIGINAL matrix, lambda_k = v_k · (A0 v_k): the diagonal of the iterated matrix
   carries the rounding of every DMMA update (about sqrt(64)·eps per round, 1e-14 after a few dozen rounds), the quotient
   only that of one product.  T = VT · A0 was written over jb.A by a chain launch; one warp per eigenvector. */
__global__ void __launch_bounds__(256) eig_rq_kernel(const EigJob* __restrict__ jobs, double* __restrict__ lam_ws, const int* __restrict__ lam_off) {
    const EigJob jb = jobs[blockIdx.y];
    double* lam = lam_ws + lam_off[blockIdx.y];
    const int n = jb.n, np = jb.np, lane = threadIdx.x & 31;
    for (int k = blockIdx.x * 8 + (threadIdx.x >> 5); k < n; k += gridDim.x * 8) {
        double s = 0.0, vv = 0.0;
        for (int j = lane; j < n; j += 32) { const double v = jb.VT[(long long)k * np + j]; s += jb.A[(long long)k * np + j] * v; vv += v * v; }
        s = warp_sum(s); vv = warp_sum(vv);
        __syncwarp();
        if (lane == 0) { lam[k] = s / vv; jb.A[(long long)k * np + k] = 1.0 / sqrt(vv); } /* lambda = v·A0 v / v·v; the scale of row k for the gather */
    }
}
/* ascending order by rank (stable on ties); row k of the output = k-th eigenvector (without the padding) */
__global__ void __launch_bounds__(256) eig_finish_kernel(const EigJob* __restrict__ jobs, const double* __restrict__ lam_ws, const int* __restrict__ lam_off,
                                                         int* __restrict__ rank_ws, const int* __restrict__ rank_off) {
    const EigJob jb = jobs[blockIdx.y];
    int* rank_of = rank_ws + rank_off[blockIdx.y];
    const double* lam = lam_ws + lam_off[blockIdx.y];
    const int n = jb.n;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
        const double di = lam[i];
        int rk = 0;
        for (int j = 0; j < n; ++j) { const double dj = lam[j]; rk += (dj < di || (dj == di && j < i)) ? 1 : 0; }
        rank_of[i] = rk;
        jb.outW[rk] = di;
    }
}
__global__ void __launch_bounds__(256) eig_gather_kernel(const EigJob* __restrict__ jobs, const int* __restrict__ rank_ws, const int* __restrict__ rank_off) {
    const EigJob jb = jobs[blockIdx.y];
    const int* rank_of = rank_ws + rank_off[blockIdx.y];
    const int n = jb.n, np = jb.np;
    const long long tot = (long long)n * n;
    for (long long e = blockIdx.x * 256ll + threadIdx.x; e < tot; e += (long long)gridDim.x * 256) {
        const int i = (int)(e / n), j = (int)(e % n);
        jb.outA[(long long)rank_of[i] * n + j] = jb.VT[(long long)i * np + j] * jb.A[(long long)i * np + i];
    }
}

int syevd_batch(Stream* st, int nblocks, const int* n, double* const* d_A, double* const* d_w) {
    if (nblocks <= 0) return 0;
    /* blocks of up to 64 states: one launch of the single-CTA Jacobi kernel — on a side stream, beside the block-Jacobi launches
       of the larger blocks (it took 3.5 ms of every truncation when it ran in front of them) */
    JacobiJob* d_small = nullptr;
    bool forked = false;
    {
        std::vector<JacobiJob> jobs;
        for (int b = 0; b < nblocks; ++b) if (n[b] > 0 && n[b] <= JAC_NMAX) jobs.push_back({d_A[b], d_w[b], n[b], 0});
        if (!jobs.empty()) {
            constexpr int smem = 2 * JAC_NMAX * JAC_LD * (int)sizeof(double);
            /* a per-DEVICE attribute: set on every call (cheap), a process may hold contexts on several devices */
            CUDA_OK(cudaFuncSetAttribute(jacobi_eig_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            if (!st->aux) {
                CUDA_OK(cudaStreamCreateWithFlags(&st->aux, cudaStreamNonBlocking));
                CUDA_OK(cudaEventCreateWithFlags(&st->ev_fork, cudaEventDisableTiming));
                CUDA_OK(cudaEventCreateWithFlags(&st->ev_join, cudaEventDisableTiming));
            }
            d_small = (JacobiJob*)malloc_bytes(st, jobs.size() * sizeof(JacobiJob));
            CUDA_OK(cudaMemcpyAsync(d_small, jobs.data(), jobs.size() * sizeof(JacobiJob), cudaMemcpyHostToDevice, st->s)); /* (pageable source: staged before the call returns) */
            CUDA_OK(cudaEventRecord(st->ev_fork, st->s));
            CUDA_OK(cudaStreamWaitEvent(st->aux, st->ev_fork, 0));
            jacobi_eig_kernel<<<(int)jobs.size(), JAC_THREADS, smem, st->aux>>>(d_small);
            LAUNCH_CHECK();
            CUDA_OK(cudaEventRecord(st->ev_join, st->aux));
            forked = true;
        }
    }
    /* the main stream continues only when the side stream is done; the job list is freed after that */
    auto join = [&]() {
        if (forked) { CUDA_OK(cudaStreamWaitEvent(st->s, st->ev_join, 0)); CUDA_OK(cudaStreamSynchronize(st->s)); free_bytes(st, d_small); forked = false; }
    };
    std::vector<int> big;
    for (int b = 0; b < nblocks; ++b) if (n[b] > JAC_NMAX) big.push_back(b);
    if (big.empty()) { join(); return 0; }
    std::stable_sort(big.begin(), big.end(), [&](int a, int b) { return n[a] > n[b]; });
    const int nj = (int)big.size();
    /* one workspace for everything: A, VT (np^2 each), Q (nb/2 x 64 x 64), flags */
    std::vector<EigJob> jobs((size_t)nj);
    size_t dbl = 0, ints = 0;
    for (int q = 0; q < nj; ++q) {
        EigJob& jb = jobs[(size_t)q];
        jb.n = n[big[q]]; jb.np = (jb.n + ET - 1) / ET * ET; jb.nb = jb.np / EB; jb.pad = 0;
        dbl += 2 * (size_t)jb.np * jb.np + (size_t)(jb.nb / 2) * ET * ET + 2 + (size_t)jb.np; /* every piece a multiple of 2 doubles: 16-byte cp.async */
        ints += (size_t)(jb.nb / 2) + 2 + (size_t)jb.n;
    }
    double* wd = (double*)malloc_bytes(st, dbl * 8);
    int* wi = (int*)malloc_bytes(st, (ints + 4 * (size_t)nj + 16) * 4);
    std::vector<int> rank_off((size_t)nj);
    std::vector<long long> lam_off((size_t)nj);
    {
        double* pd = wd; int* pi = wi;
        for (int q = 0; q < nj; ++q) {
            EigJob& jb = jobs[(size_t)q];
            jb.A = pd; pd += (size_t)jb.np * jb.np;
            jb.VT = pd; pd += (size_t)jb.np * jb.np;
            jb.Q = pd; pd += (size_t)(jb.nb / 2) * ET * ET;
            jb.norm2 = pd; pd += 2; /* one used: every piece stays a multiple of 2 doubles */
            lam_off[(size_t)q] = pd - wd; pd += jb.np;
            jb.rot = pi; pi += jb.nb / 2;
            jb.active = pi; pi += 2;
            rank_off[(size_t)q] = (int)(pi - wi); pi += jb.n;
            jb.outA = d_A[big[q]]; jb.outW = d_w[big[q]];
        }
    }
    int* d_tab = wi + ints;  /* prefix tables + rank offsets: 4*nj + 16 ints */
    EigJob* d_jobs = (EigJob*)malloc_bytes(st, (size_t)nj * sizeof(EigJob));
    CUDA_OK(cudaMemcpyAsync(d_jobs, jobs.data(), (size_t)nj * sizeof(EigJob), cudaMemcpyHostToDevice, st->s));
    constexpr int sub_smem = 2 * ET * JAC_LD * (int)sizeof(double), app_smem = 3 * ET * ELD * (int)sizeof(double);
    CUDA_OK(cudaFuncSetAttribute(eig_sub_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sub_smem));
    CUDA_OK(cudaFuncSetAttribute(eig_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, app_smem));
    eig_norm_kernel<<<nj, 1024, 0, st->s>>>(d_jobs);
    LAUNCH_CHECK();
    CUDA_OK(cudaMemcpyAsync(d_tab, rank_off.data(), (size_t)nj * 4, cudaMemcpyHostToDevice, st->s));
    eig_perm_kernel<<<dim3(4, nj), 256, 0, st->s>>>(d_jobs, wi, d_tab);
    LAUNCH_CHECK();
    eig_init_kernel<<<dim3(64, nj), 256, 0, st->s>>>(d_jobs, wi, d_tab);
    LAUNCH_CHECK();
    CUDA_OK(cudaStreamSynchronize(st->s)); /* d_tab is reused for the prefix tables below */
    int sweeps_done = 0;
    /* live jobs are a prefix-compacted copy of the job list (largest first); tables re-uploaded when a matrix finishes */
    std::vector<int> live((size_t)nj);
    for (int q = 0; q < nj; ++q) live[(size_t)q] = q;
    std::vector<EigJob> ljobs = jobs;
    EigJob* d_live = (EigJob*)malloc_bytes(st, (size_t)nj * sizeof(EigJob));
    std::vector<int> h_tab((size_t)(2 * nj + 2));
    std::vector<int> h_active((size_t)nj * 2);
    int rc = 0;
    int round = 0;
    const int max_sweeps = 40;
    while (!live.empty()) {
        const int nl = (int)live.size();
        int* sub_prefix = h_tab.data();
        int* app_prefix = h_tab.data() + nl + 1;
        sub_prefix[0] = 0; app_prefix[0] = 0;
        int maxnb = 0;
        for (int q = 0; q < nl; ++q) {
            const EigJob& jb = jobs[(size_t)live[(size_t)q]];
            ljobs[(size_t)q] = jb;
            const int npair = jb.nb / 2;
            sub_prefix[q + 1] = sub_prefix[q] + npair;
            app_prefix[q + 1] = app_prefix[q] + npair * (npair - 1) / 2 + npair * (jb.np / ET);
            maxnb = std::max(maxnb, jb.nb);
        }
        CUDA_OK(cudaMemcpyAsync(d_live, ljobs.data(), (size_t)nl * sizeof(EigJob), cudaMemcpyHostToDevice, st->s));
        CUDA_OK(cudaMemcpyAsync(d_tab, h_tab.data(), (size_t)(2 * nl + 2) * 4, cudaMemcpyHostToDevice, st->s));
        CUDA_OK(cudaStreamSynchronize(st->s)); /* host tables are reused below */
        /* one sweep of the largest live matrix (smaller ones complete at least one sweep of their own in the same rounds) */
        for (int rr = 0; rr < maxnb - 1; ++rr, ++round) {
            eig_sub_kernel<<<sub_prefix[nl], ESUB_THREADS, sub_smem, st->s>>>(d_live, d_tab, nl, round, sweeps_done == 0);
            LAUNCH_CHECK();
            eig_apply_kernel<<<app_prefix[nl], 128, app_smem, st->s>>>(d_live, d_tab + nl + 1, nl, round);
            LAUNCH_CHECK();
        }
        ++sweeps_done;
        /* which matrices went through the whole sweep without a rotation? */
        for (int q = 0; q < nl; ++q) CUDA_OK(cudaMemcpyAsync(&h_active[(size_t)q], jobs[(size_t)live[(size_t)q]].active, 4, cudaMemcpyDeviceToHost, st->s));
        CUDA_OK(cudaStreamSynchronize(st->s));
        std::vector<int> next;
        for (int q = 0; q < nl; ++q) if (h_active[(size_t)q]) next.push_back(live[(size_t)q]);
        for (int q : next) CUDA_OK(cudaMemsetAsync(jobs[(size_t)q].active, 0, 4, st->s));
        live.swap(next);
        if (round > max_sweeps * 256 || (round / std::max(1, maxnb - 1)) > max_sweeps) { if (!live.empty()) { g_err = "block Jacobi did not converge"; rc = 107; } break; }
    }
    WorkItem* d_items = nullptr;
    Segment* d_segs = nullptr;
    if (!rc) {
        /* T = VT[0:n, 0:n] · A0 over jb.A (the iterated matrix is no longer needed), on the chain kernel */
        std::vector<WorkItem> items;
        std::vector<Segment> segs;
        for (int q = 0; q < nj; ++q) {
            const EigJob& jb = jobs[(size_t)q];
            Segment sg;
            std::memset(&sg, 0, sizeof sg);
            sg.type = SEG_GEMM; sg.coef = 1.0; sg.K = jb.n;
            sg.A = jb.VT; sg.lda_m = jb.np; sg.lda_k = 1;
            sg.B = jb.outA; sg.ldb_n = 1; sg.ldb_k = jb.n;
            segs.push_back(sg);
            for (int m0 = 0; m0 < jb.n; m0 += TILE)
                for (int n0 = 0; n0 < jb.n; n0 += TILE) {
                    WorkItem it;
                    std::memset(&it, 0, sizeof it);
                    it.C = jb.A + (long long)m0 * jb.np + n0; it.ldc = jb.np; it.m0 = m0; it.n0 = n0;
                    it.tm = std::min(TILE, jb.n - m0); it.tn = std::min(TILE, jb.n - n0);
                    it.seg_begin = q; it.seg_end = q + 1;
                    items.push_back(it);
                }
        }
        d_items = (WorkItem*)malloc_bytes(st, items.size() * sizeof(WorkItem));
        d_segs = (Segment*)malloc_bytes(st, segs.size() * sizeof(Segment));
        CUDA_OK(cudaMemcpyAsync(d_items, items.data(), items.size() * sizeof(WorkItem), cudaMemcpyHostToDevice, st->s));
        CUDA_OK(cudaMemcpyAsync(d_segs, segs.data(), segs.size() * sizeof(Segment), cudaMemcpyHostToDevice, st->s));
        for (int q = 0; q < nj; ++q) h_tab[(size_t)q] = (int)lam_off[(size_t)q];
        CUDA_OK(cudaMemcpyAsync(d_tab, rank_off.data(), (size_t)nj * 4, cudaMemcpyHostToDevice, st->s));
        CUDA_OK(cudaMemcpyAsync(d_tab + nj, h_tab.data(), (size_t)nj * 4, cudaMemcpyHostToDevice, st->s));
        run_chain(st, d_items, (int)items.size(), d_segs, nullptr, nullptr, nullptr);
        eig_rq_kernel<<<dim3(16, nj), 256, 0, st->s>>>(d_jobs, wd, d_tab + nj);
        LAUNCH_CHECK();
        eig_finish_kernel<<<dim3(4, nj), 256, 0, st->s>>>(d_jobs, wd, d_tab + nj, wi, d_tab);
        LAUNCH_CHECK();
        eig_gather_kernel<<<dim3(64, nj), 256, 0, st->s>>>(d_jobs, wi, d_tab);
        LAUNCH_CHECK();
        CUDA_OK(cudaStreamSynchronize(st->s)); /* the host item lists must outlive their copies */
    }
    join();
    CUDA_OK(cudaStreamSynchronize(st->s)); /* host tables and the workspace die with this scope */
    free_bytes(st, d_items);
    free_bytes(st, d_segs);
    free_bytes(st, d_live);
    free_bytes(st, d_jobs);
    free_bytes(st, wi);
    free_bytes(st, wd);
    return rc;
}

}  // namespace dev
