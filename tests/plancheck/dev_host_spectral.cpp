/*  TEST-ONLY host emulation of dev::lanczos_batch (csrc/dev.h) — NOT part of the product.
 *
 *  The naive loops behind the spectral-function recurrence (csrc/spectral.cpp) in tests/plancheck/libdmrgx_plancheck.so, built
 *  beside dev_host.cpp so that `pytest -m "not gpu"` runs the real host logic; the product library links dev_cuda.cu's
 *  lanczos_kernel.  Same passes and stopping rules, plain sequential sums.
 */
#include <cmath>
#include <stdexcept>

#include "dev.h"

namespace dev {

int lanczos_blocks(long long) { return 1; }

void lanczos_batch(Stream*, const LanczosBatch& L, int pass, int t, const double* prev, double* cur, double* y) {
    /* lanczos_kernel strides column c by ld: shorter columns would overlap */
    if (L.nb > 0 && L.n > 0 && L.ld < L.n) throw std::runtime_error("lanczos_batch: ld below n");
    for (int col = 0; col < L.nb; ++col) {
        if (L.done[col]) continue;
        double* u = cur + (long long)col * L.ld;
        double* w = y + (long long)col * L.ld;
        const double* p = prev + (long long)col * L.ld;
        double s = 0.0;
        if (pass == 0) {
            for (long long q = 0; q < L.n; ++q) s += w[q] * w[q];
            const bool zero = s <= L.zero2[col];
            L.norm2[col] = zero ? 0.0 : s;
            if (zero) L.done[col] = 1;
            else L.scale[col] = std::sqrt(s);
        } else if (pass == 1) {
            const double c = L.scale[col];
            for (long long q = 0; q < L.n; ++q) {
                u[q] /= c;
                w[q] = w[q] / c - (t > 0 ? c * p[q] : 0.0);
                s += u[q] * w[q];
            }
            L.a[col] = s;
            L.alpha[(long long)col * L.nsteps + t] = s;
            if (t == L.nsteps - 1) { L.ndone[col] = L.nsteps; L.done[col] = 1; }
        } else {
            const double a = L.a[col];
            for (long long q = 0; q < L.n; ++q) { w[q] -= a * u[q]; s += w[q] * w[q]; }
            const double beta = std::sqrt(s), bt = t > 0 ? L.scale[col] : 0.0;
            if (beta <= LANCZOS_BETA_REL * std::sqrt(a * a + bt * bt)) { L.ndone[col] = t + 1; L.done[col] = 1; }
            else { L.beta[(long long)col * L.nsteps + t + 1] = beta; L.scale[col] = beta; }
        }
    }
}

}  // namespace dev
