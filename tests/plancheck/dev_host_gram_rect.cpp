/*  TEST-ONLY host emulation of dev::gram_rect (csrc/dev.h) — NOT part of the product.
 *
 *  The naive loop behind the Lanczos overlaps of the spectral recurrence (csrc/corr.cpp) in
 *  tests/plancheck/libdmrgx_plancheck.so, built beside dev_host.cpp so that `pytest -m "not gpu"` runs the real host logic; the
 *  product library links dev_cuda.cu's gram_kernel<true>.  Plain sums, and the alignment refusal of the device code.
 */
#include <cstdint>
#include <stdexcept>

#include "dev.h"

namespace dev {

void gram_rect(Stream*, const double* P, long long ldp, int np, const double* Q, long long ldq, int nq, long long n, double* G, long long gs,
               long long gc) {
    if (np <= 0 || nq <= 0) return;
    /* gram_kernel stages its columns with 16-byte copies */
    if ((ldp & 1) || (ldq & 1) || ((uintptr_t)P & 15) || ((uintptr_t)Q & 15))
        throw std::runtime_error("gram_rect: columns must be 16-byte aligned (P and Q aligned, ldp and ldq even)");
    for (int i = 0; i < np; ++i)
        for (int j = 0; j < nq; ++j) {
            double s = 0;
            for (long long q = 0; q < n; ++q) s += P[i * ldp + q] * Q[j * ldq + q];
            G[i * gs + j * gc] = s;
        }
}

}  // namespace dev
