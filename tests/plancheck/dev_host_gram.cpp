/*  TEST-ONLY host emulation of dev::gram (csrc/dev.h) — NOT part of the product.
 *
 *  The naive loop behind the correlation-matrix planner (csrc/corr.cpp) in tests/plancheck/libdmrgx_plancheck.so, built beside
 *  dev_host.cpp so that `pytest -m "not gpu"` runs the real planner; the product library links dev_cuda.cu's gram_kernel.
 */
#include "dev.h"

namespace dev {

void gram(Stream*, const double* P, long long ldp, int np, long long n, double* G) {
    for (int i = 0; i < np; ++i)
        for (int j = i; j < np; ++j) {
            double s = 0;
            for (long long q = 0; q < n; ++q) s += P[i * ldp + q] * P[j * ldp + q];
            G[(long long)i * np + j] = G[(long long)j * np + i] = s;
        }
}

}  // namespace dev
