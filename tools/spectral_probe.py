"""The continued-fraction recurrence of the dynamical structure factor (dmrgx_spectral_lanczos) on the 12x6 J1-J2 sweep-midpoint
superblock, against the bare superblock applies it is made of.

    python tools/spectral_probe.py [m ...] [--nsteps 64] [--json out.json]

The superblock is tools/corr_probe.py's (every site of the synthetic block carries dense Sz_i / Sp_i); psi is seeded and
normalised.  The call runs op Sz with this superblock's own Hamiltonian as the target, over the 2·72 = 144 start vectors of the
12x6 momentum grid (cos and sin parts, as the driver's -do_spectral_function builds them).  Reports the call's time (host clock
around the synchronous call, after a small warm-up call), the time of one bare dmrgx_hshell_apply on the same shell (host
clock around 50 back-to-back applies ending in a synchronise of the library's stream, after 5 warm-up ones), and the overhead
of everything else — panels, start vectors, recurrence passes, launch gaps — as the call's time over nvec·nsteps bare
applies, minus one.  The card name and power limit are read in the same run."""
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
from corr_probe import card, superblock  # noqa: E402


def momentum_coefs(Lx, Ly):
    """cos(q·r_s)/√N and sin(q·r_s)/√N for every q of the Lx×Ly grid, sites in the driver's snake order"""
    N = Lx * Ly
    xy = np.array([[s // Ly, s % Ly if (s // Ly) % 2 == 0 else Ly - 1 - s % Ly] for s in range(N)], float)
    c = []
    for kx in range(Lx):
        for ky in range(Ly):
            ph = xy @ np.array([2 * np.pi * kx / Lx, 2 * np.pi * ky / Ly])
            c += [np.cos(ph) / np.sqrt(N), np.sin(ph) / np.sqrt(N)]
    return np.array(c)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("m", type=int, nargs="*", default=[2048, 4096])
    ap.add_argument("--nsteps", type=int, default=64)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    P = dmrgx_loader.load_package()
    ctx = P.Context(0)
    name, power = card()
    ham = W.CONFIGS["j1j2_12x6"]
    coef = momentum_coefs(ham["Lx"], ham["Ly"])
    results = []
    for m in a.m:
        enl, kb, nside = superblock(P, ctx, m)
        n = 2 * nside
        terms = P.HamiltonianTerms(ham["Lx"], ham["Ly"], ham["J1"], ham["Jz1"], ham["J2"], ham["Jz2"], n, ham["bcx"], ham["bcy"])
        H = kb.KronSumConstruct(terms)
        D = kb.NumStates()
        x = np.random.default_rng(7).standard_normal(D)
        psi = ctx.vec(D, x / np.linalg.norm(x))
        kb.SpectralLanczos(psi, H, P.OpSz, coef[:2], 4)               # warm-up (module load, heap growth)
        l0 = P.launch_count()
        t0 = time.perf_counter()
        r = kb.SpectralLanczos(psi, H, P.OpSz, coef, a.nsteps)       # synchronous: returns after the last batch's copies
        call_s = time.perf_counter() - t0
        launches = P.launch_count() - l0
        # one bare apply on the same shell
        y = ctx.vec(D)
        for _ in range(5):
            H.MatMult(psi, y)
        ctx.sync()
        t0 = time.perf_counter()
        for _ in range(50):
            H.MatMult(psi, y)
        ctx.sync()
        apply_ms = (time.perf_counter() - t0) * 1e3 / 50
        nvec = len(coef)
        applies_s = nvec * a.nsteps * apply_ms * 1e-3
        res = dict(m=m, D=D, sites=n, nvec=nvec, nsteps=a.nsteps, call_s=call_s, apply_ms=apply_ms, applies_s=applies_s,
                   overhead=call_s / applies_s - 1.0, launches=launches, flops=r["flops"], tflops=r["flops"] / call_s / 1e12,
                   steps_done_min=int(r["nsteps_done"].min()), steps_done_max=int(r["nsteps_done"].max()),
                   finite=bool(np.isfinite(r["alpha"]).all() and np.isfinite(r["beta"]).all()), card=name, power_limit=power)
        print(json.dumps(res))
        results.append(res)
        del H, psi, y, kb, enl
    if a.json:
        json.dump(results, open(a.json, "w"), indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
