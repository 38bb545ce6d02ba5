/*  TEST-ONLY shim over dev::gram_rect (csrc/dev.h) for tests/test_dynamical_correlations.py — NOT part of the product.
 *
 *  The conventions of tests/devcheck/devcheck.cpp, in a library of its own: each host array is [guard | payload | guard] and
 *  goes to the device and back whole, so the test sees what the kernel did to the guards; a guard below 4 KiB or below one
 *  leading dimension is refused.  Built twice (csrc/Makefile): libdevcheck_gram_rect_host.so over the host emulation
 *  (tests/plancheck/dev_host*.cpp), libdevcheck_gram_rect_cuda.so over the product's own sm_100a object build/dev_cuda.o.
 *  Every entry point returns 0 or -1; dc_error() holds the message (a refusal of the shim, or what dev:: threw).
 */
#include <cstdio>
#include <stdexcept>
#include <string>

#include "dev.h"

namespace {

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
struct Buf {
    double* host = nullptr;
    double* dev_base = nullptr;
    long long total = 0, guard = 0;
    bool out = false;
    Buf() = default;
    Buf(const Buf&) = delete;
    void set(double* h, long long tot, long long g, long long need, long long ld, bool is_out, const char* name) {
        REFUSE_IF(!h, "%s is NULL", name);
        REFUSE_IF(g < MIN_GUARD || g < ld || (g & 1), "%s: guard of %lld elements is below 4 KiB, below the leading dimension %lld, or odd", name, g, ld);
        REFUSE_IF(need < 0 || tot < 2 * g + need, "%s: %lld elements hold no %lld-element payload between two %lld-element guards", name, tot, need, g);
        host = h; total = tot; guard = g; out = is_out;
        dev_base = (double*)dev::malloc_bytes(stream(), sizeof(double) * (size_t)tot);
        dev::h2d(stream(), dev_base, host, sizeof(double) * (size_t)tot);
    }
    double* p() const { return dev_base + guard; }
    void back() { if (out) dev::d2h(stream(), host, dev_base, sizeof(double) * (size_t)total); }
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

}  // namespace

extern "C" {

const char* dc_error() { return g_msg.c_str(); }

/* G[i·gs + j·gc] = (PᵀQ)[i][j]: P holds np columns of ldp doubles, Q nq columns of ldq; `shift` moves both column bases by
   that many doubles (alignment checks) */
int dc_gram_rect(double* P, long long nP, long long ldp, int np, double* Q, long long nQ, long long ldq, int nq, long long n, int shift, double* G,
                 long long nG, long long gs, long long gc, long long guard) {
    return guarded([&] {
        REFUSE_IF(np < 1 || nq < 1 || n < 0 || ldp < n || ldq < n || shift < 0 || shift > 1 || gs < 0 || gc < 0, "np, nq, n, ldp, ldq, shift or strides");
        Buf p, q, g;
        p.set(P, nP, guard, (np - 1) * ldp + n + shift, ldp, false, "P");
        q.set(Q, nQ, guard, (nq - 1) * ldq + n + shift, ldq, false, "Q");
        g.set(G, nG, guard, (np - 1) * gs + (nq - 1) * gc + 1, 0, true, "G");
        dev::gram_rect(stream(), p.p() + shift, ldp, np, q.p() + shift, ldq, nq, n, g.p(), gs, gc);
        g.back();
        dev::sync(stream());
    });
}

}  // extern "C"
