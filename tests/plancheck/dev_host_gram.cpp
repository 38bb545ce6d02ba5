/*  TEST-ONLY host emulation of dev::gram (csrc/dev.h) — NOT part of the product.
 *
 *  The naive loop behind the correlation-matrix planner (csrc/corr.cpp) in tests/plancheck/libdmrgx_plancheck.so, built beside
 *  dev_host.cpp so that `pytest -m "not gpu"` runs the real planner; the product library links dev_cuda.cu's gram_kernel.
 */
#include <cstdint>
#include <stdexcept>

#include "dev.h"

namespace dev {

void gram(Stream*, const double* P, long long ldp, int np, long long n, double* G) {
    if (np <= 0 || n <= 0) {
        for (long long e = 0; e < (long long)np * np; ++e) G[e] = 0.0;
        return;
    }
    /* gram_kernel stages its columns with 16-byte copies */
    if ((ldp & 1) || ((uintptr_t)P & 15)) throw std::runtime_error("gram: columns must be 16-byte aligned (P aligned, ldp even)");
    for (int i = 0; i < np; ++i)
        for (int j = i; j < np; ++j) {
            double s = 0;
            for (long long q = 0; q < n; ++q) s += P[i * ldp + q] * P[j * ldp + q];
            G[(long long)i * np + j] = G[(long long)j * np + i] = s;
        }
}

}  // namespace dev
