"""The all-pairs spin correlation matrix (dmrgx_corr_matrix) on the 12x6 J1-J2 sweep-midpoint superblock, against the
per-correlator path (dmrgx_hshell_create_product + dmrgx_expect per entry) it replaces.

    python tools/corr_probe.py [m ...] [--reps 10] [--sample 240] [--json out.json]

Every site of the synthetic block carries dense Sz_i / Sp_i (bench_workload.synth_block_host with all sites used): the
default workload leaves the sites no Hamiltonian term touches empty, which would make their panels free.  psi is seeded
and normalised.  Reports the batched call's time (host clock around the synchronous call, after a warm-up call), its
algorithmic flops and rate, that rate as a fraction of a float64 matmul measured in the same run (torch, as bench.py
does), the card name and power limit, and the per-correlator path timed on a fixed seeded sample of same-block and
cross-block entries, extrapolated to all 3n² + n entries; the sampled entries must agree to 1e-12·max|C|."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import dmrgx_loader  # noqa: E402
import bench_workload as W  # noqa: E402
from bench import fp64_peak_tflops  # noqa: E402
from test_correlation_matrix import per_correlator, SM, SZ, SP  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in out.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:  # the numbers stay usable without the label
        return "unknown (%s)" % e, "unknown"


def superblock(P, ctx, m):
    ham = W.CONFIGS["j1j2_12x6"]
    N = ham["Lx"] * ham["Ly"]
    nblk = N // 2 - 1
    T = lambda k: P.HamiltonianTerms(ham["Lx"], ham["Ly"], ham["J1"], ham["Jz1"], ham["J2"], ham["Jz2"], k, ham["bcx"], ham["bcy"])
    host = W.synth_block_host(m, nblk, set(range(nblk)))
    blk = P.Block.Initialize(ctx, nblk, host["qn"], host["sizes"])
    for i in range(nblk):
        blk.set_operator(P.OpSz, i, *host["ops"][("Sz", i)])
        blk.set_operator(P.OpSp, i, *host["ops"][("Sp", i)])
    blk.set_operator(P.OpH, 0, *host["ops"]["H"])
    enl = P.KronEye_Explicit(blk, P.Block.SingleSite(ctx), T(nblk + 1))
    return enl, P.KronBlocks(enl, enl, [0.0]), nblk + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("m", type=int, nargs="*", default=[2048, 4096])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sample", type=int, default=240)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert a.reps >= 10 and a.sample >= 200
    import torch
    P = dmrgx_loader.load_package()
    ctx = P.Context(0)
    name, power = card()
    peak = fp64_peak_tflops(torch, torch.device("cuda:0"))
    results = []
    for m in a.m:
        enl, kb, nside = superblock(P, ctx, m)
        n = 2 * nside
        D = kb.NumStates()
        x = np.random.default_rng(7).standard_normal(D)
        psi = ctx.vec(D, x / np.linalg.norm(x))
        l0 = P.launch_count()
        got = kb.CorrelationMatrix(psi)                       # warm-up (module load, heap growth)
        launches = P.launch_count() - l0
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            kb.CorrelationMatrix(psi)                         # synchronous: returns after the device-to-host copy
            ts.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.median(ts))
        tflops = got["flops"] / (ms * 1e-3) / 1e12
        # the per-correlator path on a fixed seeded sample: half same-block, half cross-block pairs
        rng = np.random.default_rng(11)
        names = {"SzSz": (SZ, SZ), "SpSm": (SP, SM), "SmSp": (SM, SP)}
        sample = []
        while len(sample) < a.sample:
            i = int(rng.integers(n))
            j = int(rng.integers(nside)) + (0 if (len(sample) % 2 == 0) == (i < nside) else nside)
            sample.append((list(names)[len(sample) % 3], i, j))
        cmax = max(np.abs(got[k]).max() for k in names)
        per_correlator(P, kb, psi, nside, nside, *(sample[0][1], names[sample[0][0]][0], sample[0][2], names[sample[0][0]][1]))  # warm-up
        worst = 0.0
        t0 = time.perf_counter()
        for k, i, j in sample:
            v = per_correlator(P, kb, psi, nside, nside, i, names[k][0], j, names[k][1])
            worst = max(worst, abs(v - got[k][i, j]))
        per_entry = (time.perf_counter() - t0) / len(sample)
        r = dict(m=m, D=D, sites=n, launches=launches, ms=ms, ms_min=1e3 * min(ts), flops=got["flops"], tflops=tflops, fp64_matmul_tflops=peak,
                 frac_of_fp64_matmul=tflops / peak, per_correlator_ms=1e3 * per_entry, per_correlator_all_s=per_entry * (3 * n * n + n),
                 speedup=per_entry * (3 * n * n + n) / (ms * 1e-3), sample=len(sample), sample_max_abs_diff=worst, max_abs_C=cmax,
                 agree=bool(worst <= 1e-12 * cmax), card=name, power_limit=power)
        print(json.dumps(r))
        assert r["agree"], r
        results.append(r)
        del got, psi, kb, enl
    if a.json:
        json.dump(results, open(a.json, "w"), indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
