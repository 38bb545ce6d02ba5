"""The all-pairs spin correlation matrix (dmrgx_corr_matrix, KronBlocks.CorrelationMatrix) and the driver's
-do_correlation_matrix output.  Every check runs on the host emulation of the device layer (tests/plancheck) and, under
-m gpu, on the CUDA library."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import driver_common as dc
from measure_common import (HEIS_CHAIN12, J1J2_CYL, SM, SP, SZ, P, ctx, exact_diagonalisation, exact_halves, exe,  # noqa: F401
                            ham_terms, ngpus, oracle_blocks, product_expect, random_psi)


# ---- references --------------------------------------------------------------------------------------------------------

def exact_correlators(terms, N):
    """ground-state energy of the lattice Hamiltonian in the Sz = 0 sector, the gap above it and every two-point correlator"""
    w, psi, _, ops, _ = exact_diagonalisation(terms, N, k=2)
    apply = {k: ops[k] @ psi for k in ops}
    out = dict(SzSz=np.zeros((N, N)), SpSm=np.zeros((N, N)), SmSp=np.zeros((N, N)), Sz=np.array([psi @ apply[(SZ, i)] for i in range(N)]))
    for i in range(N):
        for j in range(N):
            out["SzSz"][i, j] = apply[(SZ, i)] @ apply[(SZ, j)]
            out["SpSm"][i, j] = apply[(SM, i)] @ apply[(SM, j)]
            out["SmSp"][i, j] = apply[(SP, i)] @ apply[(SP, j)]
    return w[0], w[1] - w[0], out


def energy_from(C_, terms):
    key = {(SZ, SZ): "SzSz", (SP, SM): "SpSm", (SM, SP): "SmSp"}
    return sum(a * C_[key[(io, jo)]][i, j] for (a, io, i, jo, j) in terms)


# ---- the library ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", ["L=R", "L!=R", "spin1"])
def test_every_entry_matches_the_per_correlator_path(P, ctx, orc, case):
    """Oracle warm-up blocks of the 4x4 J1-J2 cylinder: all 3n² + n entries equal dmrgx_hshell_create_product + dmrgx_expect
    for the same operator lists (same-block entries are products of the block's own operators in list order)."""
    nL, nR, spin = {"L=R": (8, 8, 1), "L!=R": (8, 6, 1), "spin1": (8, 8, 2)}[case]
    pL, pR = oracle_blocks(orc, P, ctx, nL, nR, spin)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 17)
    got = kb.CorrelationMatrix(dpsi)
    n = nL + nR
    assert got["SzSz"].shape == (n, n) and got["Sz"].shape == (n,) and got["flops"] > 0
    worst = 0.0
    for i in range(n):
        worst = max(worst, abs(got["Sz"][i] - product_expect(P, kb, dpsi, nL, n, [(SZ, i)])))
        for j in range(n):
            for name, oi, oj in (("SzSz", SZ, SZ), ("SpSm", SP, SM), ("SmSp", SM, SP)):
                worst = max(worst, abs(got[name][i, j] - product_expect(P, kb, dpsi, nL, n, [(oi, i), (oj, j)])))
    assert worst < 1e-12, worst


def _check_exact(P, ctx, ham):
    blk, terms = exact_halves(P, ctx, ham)
    kb = P.KronBlocks(blk, blk, [0.0])
    e0, psi, st = kb.KronSumConstruct(terms).EPSSolve(tol=1e-12)
    assert st["converged"]
    got = kb.CorrelationMatrix(psi)
    N = ham["Lx"] * ham["Ly"]
    e_ed, gap, ref = exact_correlators(terms, N)
    assert gap > 1e-6 and abs(e0 - e_ed) < 1e-9 * abs(e_ed)
    for k in ("SzSz", "SpSm", "SmSp", "Sz"):
        assert np.abs(got[k] - ref[k]).max() < 1e-8, (k, np.abs(got[k] - ref[k]).max())
    assert abs(energy_from(got, terms) - e0) <= 1e-10 * abs(e0)


def test_exact_blocks_match_exact_diagonalisation_chain12(P, ctx):
    """Un-truncated 6-site halves of the 12-site open Heisenberg chain: the matrices equal scipy ED in the Sz = 0 sector and
    Σ_terms a·C reproduces the ground-state energy."""
    _check_exact(P, ctx, HEIS_CHAIN12)


@pytest.mark.gpu
def test_exact_blocks_match_exact_diagonalisation_j1j2_4x4(P, ctx):
    if P.kind != "cuda":
        pytest.skip("16-site ED against the CUDA library only")
    _check_exact(P, ctx, J1J2_CYL)


def test_sum_rules_under_truncation(P, ctx, orc):
    """Rotations conserve Sz, so on truncated blocks Σ_i Sz_i = qn and Σ_ij SzSz_ij = qn² for a normalised psi of sector qn;
    in the top sector there is nothing for S+ to reach and SmSp is zero."""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 6)
    for qn in (0.0, 1.0):
        kb = P.KronBlocks(pL, pR, [qn])
        got = kb.CorrelationMatrix(random_psi(ctx, kb.NumStates(), 3)[0])
        assert abs(got["Sz"].sum() - qn) < 1e-10
        assert abs(got["SzSz"].sum() - qn * qn) < 1e-10
    top = max(pL.sectors()[0]) + max(pR.sectors()[0])
    kb = P.KronBlocks(pL, pR, [top])
    got = kb.CorrelationMatrix(random_psi(ctx, kb.NumStates(), 4)[0])
    assert not got["SmSp"].any() and np.abs(got["SpSm"]).max() > 0


def test_errors(P, ctx, orc):
    """62: psi NULL; 56: not exactly one sector; 73: a block without Sz_i / Sp_i, the site named in the message."""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 8)
    kb = P.KronBlocks(pL, pR, [0.0])
    with pytest.raises(P.DmrgxError) as e:
        kb.CorrelationMatrix(None)
    assert e.value.code == 62
    for qns in ([], [0.0, 1.0]):
        k2 = P.KronBlocks(pL, pR, qns)
        with pytest.raises(P.DmrgxError) as e:
            k2.CorrelationMatrix(ctx.vec(k2.NumStates(), np.ones(k2.NumStates())))
        assert e.value.code == 56
    b = P.Block.Initialize(ctx, 2, [1.0, 0.0, -1.0], [1, 2, 1])
    empty = (np.zeros(5, np.int64), np.zeros(0, np.int64), np.zeros(0))
    b.set_operator(P.OpSz, 0, *empty)
    b.set_operator(P.OpSp, 0, *empty)
    k3 = P.KronBlocks(b, P.Block.SingleSite(ctx), [0.5])
    with pytest.raises(P.DmrgxError) as e:
        k3.CorrelationMatrix(ctx.vec(k3.NumStates(), np.ones(k3.NumStates())))
    assert e.value.code == 73 and "site 1" in str(e.value)


@pytest.mark.gpu
def test_two_calls_are_bitwise_equal(P, ctx):
    """the Gram reduction sums its row slabs in a fixed order: no run-to-run noise (4x4 J1-J2, D = 12870, two slabs)"""
    if P.kind != "cuda":
        pytest.skip("the CUDA kernels only")
    blk, _ = exact_halves(P, ctx, J1J2_CYL)
    kb = P.KronBlocks(blk, blk, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 9)
    a, b = kb.CorrelationMatrix(dpsi), kb.CorrelationMatrix(dpsi)
    for k in ("SzSz", "SpSm", "SmSp", "Sz"):
        assert np.array_equal(a[k], b[k]), k


# ---- the driver ----------------------------------------------------------------------------------------------------------

# (arguments, lattice, mwarmup, msweeps, exact): `exact` runs never truncate a block (2^6 = 64 states on the 12-site chain), so the
# matrices hold the lattice energy exactly.  Under truncation, intra-block terms become products of projected operators, which
# differ from the projected products in the block Hamiltonian: Σ a·C is then not the step energy (the 4x4 sweep at m = 256
# truncates the 13-site blocks of the sweep's first half).
CHAIN12_RUN = (["-Lx", 12, "-Ly", 1, "-heisenberg", 1, "-BCopen"], HEIS_CHAIN12, 64, [64], True)
DRIVER_CASES = {"plancheck": [CHAIN12_RUN],
                "cuda": [(["-Lx", 4, "-Ly", 4, "-J1", 0.5, "-Jz1", 1, "-J2", 0.25, "-Jz2", 0.5], J1J2_CYL, 256, [256], False), CHAIN12_RUN]}


def check_records(P, recs, docs, ham, exact):
    N = ham["Lx"] * ham["Ly"]
    terms = ham_terms(P, ham, N)
    corr = docs["Correlations"]
    names = [c["name"] for c in corr["info"]]
    assert len(recs) == len(corr["values"]) >= 2
    steps = {row[0]: row[-1] for row in docs["DMRGSteps"]["table"]}
    for rec, vals in zip(recs, corr["values"]):
        M = {k: np.array(rec[k]) for k in ("SzSz", "SpSm", "SmSp", "Sz")}
        assert M["SzSz"].shape == (N, N) and len(rec["sites"]) == N
        for name, v in zip(names, vals):
            if name.startswith("NearestNeighborSzSz"):
                i, j = (int(t) for t in name.split("(")[1].split(")")[0].split())
                assert abs(M["SzSz"][i, j] - v) <= 1e-5 * abs(v) + 1e-12, (name, M["SzSz"][i, j], v)
        if exact:
            e = steps[rec["GlobIdx"]]
            assert abs(energy_from(M, terms) - e) <= 1e-9 * abs(e)
        xy = np.array(rec["sites"], float)
        Css = M["SzSz"] + 0.5 * (M["SpSm"] + M["SmSp"])
        for kx in range(ham["Lx"]):
            for ky in range(ham["Ly"]):
                q = np.array([2 * np.pi * kx / ham["Lx"], 2 * np.pi * ky / ham["Ly"]])
                ph = xy @ q
                s = np.sum(np.cos(ph[:, None] - ph[None, :]) * Css) / N
                assert abs(rec["StructureFactor"][kx][ky] - s) < 1e-12


def test_driver_writes_the_matrix_at_every_measurement(P, exe, tmp_path):
    """-do_correlation_matrix 1: one record per Correlations.json row, consistent with the nearest-neighbour correlators,
    with the step's energy (on exact blocks) and with its own structure factor; without the option there is no file and the other outputs
    are byte for byte those of the run with it."""
    for k, (args, ham, mw, ms, exact) in enumerate(DRIVER_CASES[P.kind]):
        docs, _ = dc.run_driver(exe, tmp_path / ("with%d" % k), args, mw, ms, extra=["-do_correlation_matrix", "1"])
        out = str(tmp_path / ("with%d" % k) / "data") + "/"
        recs = json.load(open(out + "CorrelationMatrix.json"))
        check_records(P, recs, docs, ham, exact)
        dc.run_driver(exe, tmp_path / ("without%d" % k), args, mw, ms)
        out0 = str(tmp_path / ("without%d" % k) / "data") + "/"
        assert not os.path.exists(out0 + "CorrelationMatrix.json")
        for f in ("DMRGSteps", "EntanglementSpectra", "Correlations"):
            assert open(out + f + ".json", "rb").read() == open(out0 + f + ".json", "rb").read(), f


@pytest.mark.gpu
@pytest.mark.skipif(ngpus() < 2, reason="needs two GPUs")
def test_two_rank_driver_writes_the_same_matrix(P, exe, tmp_path):
    if P.kind != "cuda":
        pytest.skip("the CUDA executable only")
    args, ham, mw, ms, _ = DRIVER_CASES["cuda"][0]
    one, _ = dc.run_driver(exe, tmp_path / "one", args, mw, ms, extra=["-do_correlation_matrix", "1"])
    out = str(tmp_path / "two") + "/"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--no-python", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", exe] + [str(a) for a in args] + ["-mwarmup", str(mw), "-msweeps", ",".join(map(str, ms)), "-H_eps_tol", "1e-12",
                                                                       "-do_correlation_matrix", "1", "-data_dir", out]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    a = json.load(open(str(tmp_path / "one" / "data") + "/CorrelationMatrix.json"))
    b = json.load(open(out + "CorrelationMatrix.json"))
    assert len(a) == len(b)
    for x, y in zip(a, b):
        for k in ("SzSz", "SpSm", "SmSp", "Sz", "StructureFactor"):
            assert np.abs(np.array(x[k]) - np.array(y[k])).max() < 1e-10, k
