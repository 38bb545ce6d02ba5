"""The real-space dynamical correlation matrix (dmrgx_spectral_lanczos_overlaps) on the 12x6 J1-J2 sweep-midpoint superblock,
against the same recurrence without overlaps and against the 144-vector momentum-grid call of the spectral function.

    python tools/dyncorr_probe.py [m ...] [--nsteps 64] [--json out.json]

The superblock is tools/corr_probe.py's (every site of the synthetic block carries dense Sz_i / Sp_i); psi is seeded and
normalised.  All calls run op Sz with this superblock's own Hamiltonian as the target and nsteps steps:
  - overlaps: the 72 single-site sources (coef = I) through dmrgx_spectral_lanczos_overlaps;
  - plain:    the same 72 sources through dmrgx_spectral_lanczos;
  - q-grid:   the 144 cos / sin start vectors of the 12x6 momentum grid (tools/spectral_probe.py) through dmrgx_spectral_lanczos.
Each is timed with a host clock around the synchronous call, after a small warm-up call, in the order overlaps, plain, q-grid,
overlaps, plain (the two repeats give the spread).  The gram_rect kernels are timed apart, in a torch.profiler run of a short
overlaps call (72 sources, 4 steps): the summed device time of gram_kernel<true> and gram_rect_reduce_kernel per (batch, step).
Their bound is max(2·n·nb·D / DGEMM rate, (n + nb)·D·8 bytes / copy rate), with the FP64 rate of a cuBLAS DGEMM and the rate of
a 2 GiB device-to-device copy measured in the same run (measurement tools only, never the product's path).  The card name and
power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import dmrgx_loader  # noqa: E402
import bench_workload as W  # noqa: E402
from bench import fp64_peak_tflops  # noqa: E402
from corr_probe import card, superblock  # noqa: E402
from spectral_probe import momentum_coefs  # noqa: E402

SPECTRAL_BATCH_BYTES = 2.0 * 2 ** 30   # csrc/corr.cpp: device memory of the three recurrence columns of a batch


def copy_rate(torch):
    """bytes read + written per second of a 2 GiB device-to-device copy, best of 5"""
    n = 2 ** 28
    a = torch.ones(n, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n * 8 / (best * 1e-3)


def timed(f):
    t0 = time.perf_counter()
    r = f()
    return time.perf_counter() - t0, r


def gram_rect_device_ms(torch, f):
    """summed device time (ms) of the gram_rect kernels in one call of f, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    tot, count = 0.0, 0
    for e in prof.events():
        name = e.name
        if "gram_rect_reduce_kernel" in name or ("gram_kernel" in name and "true" in name):
            tot += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
            count += 1
    return tot * 1e-3, count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("m", type=int, nargs="*", default=[2048, 4096])
    ap.add_argument("--nsteps", type=int, default=64)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch
    P = dmrgx_loader.load_package()
    ctx = P.Context(0)
    name, power = card()
    dgemm = fp64_peak_tflops(torch, torch.device("cuda:0")) * 1e12
    copy = copy_rate(torch)
    ham = W.CONFIGS["j1j2_12x6"]
    qcoef = momentum_coefs(ham["Lx"], ham["Ly"])
    results = []
    for m in a.m:
        enl, kb, nside = superblock(P, ctx, m)
        n = 2 * nside
        terms = P.HamiltonianTerms(ham["Lx"], ham["Ly"], ham["J1"], ham["Jz1"], ham["J2"], ham["Jz2"], n, ham["bcx"], ham["bcy"])
        H = kb.KronSumConstruct(terms)
        D = kb.NumStates()
        x = np.random.default_rng(7).standard_normal(D)
        psi = ctx.vec(D, x / np.linalg.norm(x))
        src = np.eye(n)
        kb.SpectralLanczos(psi, H, P.OpSz, src[:2], 4, overlaps=True)   # warm-up (module load, heap growth)
        kb.SpectralLanczos(psi, H, P.OpSz, src[:2], 4)
        t_ov, r_ov = timed(lambda: kb.SpectralLanczos(psi, H, P.OpSz, src, a.nsteps, overlaps=True))
        t_plain, r_plain = timed(lambda: kb.SpectralLanczos(psi, H, P.OpSz, src, a.nsteps))
        t_q, r_q = timed(lambda: kb.SpectralLanczos(psi, H, P.OpSz, qcoef, a.nsteps))
        t_ov2, _ = timed(lambda: kb.SpectralLanczos(psi, H, P.OpSz, src, a.nsteps, overlaps=True))
        t_plain2, _ = timed(lambda: kb.SpectralLanczos(psi, H, P.OpSz, src, a.nsteps))
        same = all(np.array_equal(r_ov[k], r_plain[k]) for k in ("alpha", "beta", "norm2", "nsteps_done"))
        nb = int(max(1, min(n, SPECTRAL_BATCH_BYTES // (24 * ((D + 1) & ~1)))))
        nbatch = -(-n // nb)
        psteps = 4
        gr_ms, gr_launches = gram_rect_device_ms(torch, lambda: kb.SpectralLanczos(psi, H, P.OpSz, src, psteps, overlaps=True))
        per_step_ms = gr_ms / (nbatch * psteps)
        # the bound of one full batch's step (the last batch may be smaller)
        flops, nbytes = 2.0 * n * nb * D, (n + nb) * D * 8.0
        bound_ms = max(flops / dgemm, nbytes / copy) * 1e3
        res = dict(m=m, D=D, sites=n, nsteps=a.nsteps, batch=nb, batches=nbatch, overlaps_s=[t_ov, t_ov2], plain_s=[t_plain, t_plain2],
                   qgrid_s=t_q, overlaps_over_plain=min(t_ov, t_ov2) / min(t_plain, t_plain2) - 1.0, recurrence_bits_equal=same,
                   gram_rect_ms_per_step=per_step_ms, gram_rect_launches=gr_launches, gram_rect_bound_ms=bound_ms,
                   gram_rect_flops=flops, gram_rect_bytes=nbytes, dgemm_tflops=dgemm / 1e12, copy_gbs=copy / 1e9,
                   steps_done_min=int(r_ov["nsteps_done"].min()), steps_done_max=int(r_ov["nsteps_done"].max()),
                   finite=bool(np.isfinite(r_ov["overlaps"]).all()), card=name, power_limit=power)
        print(json.dumps(res))
        results.append(res)
        del H, psi, kb, enl
    if a.json:
        json.dump(results, open(a.json, "w"), indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
