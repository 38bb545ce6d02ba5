"""The dimer correlation matrix (dmrgx_dimer_matrix) on the 12x6 J1-J2 sweep-midpoint superblock over the 138
nearest-neighbour bonds of the cylinder, against the per-correlator path (9 four-operator dmrgx_hshell_create_product +
dmrgx_expect per entry) it replaces.

    python tools/dimer_probe.py [m ...] [--reps 10] [--sample 40] [--json out.json]

The superblock is the one of tools/corr_probe.py: every site of the synthetic block carries dense Sz_i / Sp_i, and psi is
seeded and normalised.  Reports the batched call's time (median of synchronous calls after a warm-up call, host clock),
its algorithmic flops and rate, that rate as a fraction of a float64 matmul measured in the same run, the kernel
launches of one call, the card name and power limit, and the per-correlator path timed on a fixed seeded sample of
entries <D_a psi, D_b psi>, extrapolated to all nb² + nb entries; the sampled entries must agree to 1e-12·max|DD|."""
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
from measure_common import nn_bonds, per_correlator_dimer  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("m", type=int, nargs="*", default=[2048, 4096])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--sample", type=int, default=40)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert a.reps >= 10 and a.sample >= 20
    import torch
    P = dmrgx_loader.load_package()
    ctx = P.Context(0)
    name, power = card()
    peak = fp64_peak_tflops(torch, torch.device("cuda:0"))
    ham = W.CONFIGS["j1j2_12x6"]
    bonds = [p for p, _, _ in nn_bonds(ham)]
    nb = len(bonds)
    results = []
    for m in a.m:
        enl, kb, nside = superblock(P, ctx, m)
        D = kb.NumStates()
        x = np.random.default_rng(7).standard_normal(D)
        psi = ctx.vec(D, x / np.linalg.norm(x))
        l0 = P.launch_count()
        got = kb.DimerMatrix(psi, bonds)                      # warm-up (module load, heap growth)
        launches = P.launch_count() - l0
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            kb.DimerMatrix(psi, bonds)                        # synchronous: returns after the device-to-host copy
            ts.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.median(ts))
        tflops = got["flops"] / (ms * 1e-3) / 1e12
        # the per-correlator path on a fixed seeded sample of (a, b), a few of them <D_a> (b = None)
        rng = np.random.default_rng(11)
        sample = [(int(rng.integers(nb)), None if k % 10 == 0 else int(rng.integers(nb))) for k in range(a.sample)]
        dmax = np.abs(got["DD"]).max()
        per_correlator_dimer(P, kb, psi, nside, 2 * nside, bonds[0], bonds[1])  # warm-up
        worst = 0.0
        t0 = time.perf_counter()
        for i, j in sample:
            v = per_correlator_dimer(P, kb, psi, nside, 2 * nside, bonds[i], None if j is None else bonds[j])
            worst = max(worst, abs(v - (got["D"][i] if j is None else got["DD"][i, j])))
        t_sample = time.perf_counter() - t0
        nprod = sum(3 if j is None else 9 for _, j in sample)
        per_entry = t_sample / nprod * 9                      # a full <D_a D_b> entry: 9 products
        all_s = t_sample / nprod * (9 * nb * nb + 3 * nb)
        r = dict(m=m, D=D, bonds=nb, launches=launches, ms=ms, ms_min=1e3 * min(ts), flops=got["flops"], tflops=tflops,
                 fp64_matmul_tflops=peak, frac_of_fp64_matmul=tflops / peak, per_correlator_ms_per_entry=1e3 * per_entry,
                 per_correlator_ms_per_product=1e3 * t_sample / nprod, per_correlator_all_s=all_s, speedup=all_s / (ms * 1e-3),
                 sample=len(sample), sample_max_abs_diff=worst, max_abs_DD=dmax, agree=bool(worst <= 1e-12 * dmax), card=name,
                 power_limit=power)
        print(json.dumps(r), flush=True)
        assert r["agree"], r
        results.append(r)
        del got, psi, kb, enl
    if a.json:
        json.dump(results, open(a.json, "w"), indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
