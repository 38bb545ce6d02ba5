"""The dimer (bond–bond) correlation matrix (dmrgx_dimer_matrix, KronBlocks.DimerMatrix) and the driver's -do_dimer_matrix
output.  Every check runs on the host emulation of the device layer (tests/plancheck) and, under -m gpu, on the CUDA
library."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import driver_common as dc
from measure_common import (DRIVER_M, DRIVER_RUN, HEIS_CHAIN12, J1J2_CYL, SM, SP, SZ, P, ctx,  # noqa: F401
                            exact_diagonalisation, exact_halves, exe, ham_terms, nn_bonds, oracle_blocks,
                            per_correlator_dimer, random_psi)


# ---- references --------------------------------------------------------------------------------------------------------

def lattice_pairs(P, ham, n):
    """distinct (i, j), i < j, of the lattice's Sz·Sz terms with both sites below n, split into nearest (Jz1) and next-nearest (Jz2)"""
    terms = ham_terms(P, ham, ham["Lx"] * ham["Ly"])
    nn, nnn = [], []
    for a, io, i, jo, j in terms:
        if io != SZ or max(i, j) >= n:
            continue
        p = (min(i, j), max(i, j))
        dst = nn if a == ham["Jz1"] else nnn
        if p not in dst:
            dst.append(p)
    return nn, nnn


def mixed_bonds(P, nL, n):
    """left-left, cross and right-right bonds of the 4x4 J1-J2 cylinder, nearest and next-nearest, two of them listed as (j, i)"""
    nn, nnn = lattice_pairs(P, J1J2_CYL, n)
    kind = lambda p: (p[0] >= nL) + (p[1] >= nL)
    bonds = []
    for pairs in (nn, nnn):
        for k in (0, 1, 2):
            bonds += [p for p in pairs if kind(p) == k][:1]
    bonds.append([p for p in nn if kind(p) == 1][1])
    assert {kind(p) for p in bonds} == {0, 1, 2}
    bonds[1] = bonds[1][::-1]
    bonds[4] = bonds[4][::-1]
    return bonds


def exact_dimers(terms, N, bonds):
    """exact diagonalisation in the Sz = 0 sector: ground-state energy, gap, <D_a D_b> and <D_a>"""
    w, psi, _, ops, _ = exact_diagonalisation(terms, N, k=2)
    bond_op = lambda i, j: ops[(SZ, i)] @ ops[(SZ, j)] + 0.5 * (ops[(SP, i)] @ ops[(SM, j)] + ops[(SM, i)] @ ops[(SP, j)])
    Dpsi = np.array([bond_op(i, j) @ psi for i, j in bonds])
    return w[0], w[1] - w[0], Dpsi @ Dpsi.T, Dpsi @ psi


# ---- the library ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", ["L=R", "L!=R", "spin1"])
def test_every_entry_matches_the_per_correlator_path(P, ctx, orc, case):
    """Oracle warm-up (truncated) blocks of the 4x4 J1-J2 cylinder: every <D_a psi, D_b psi> and <D_a> equals the sum of its 9
    (or 3) dmrgx_hshell_create_product + dmrgx_expect terms, for left-left, cross and right-right, nearest and next-nearest
    bonds, some given as (j, i)."""
    nL, nR, spin = {"L=R": (8, 8, 1), "L!=R": (8, 6, 1), "spin1": (8, 8, 2)}[case]
    pL, pR = oracle_blocks(orc, P, ctx, nL, nR, spin)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 17)
    n = nL + nR
    bonds = mixed_bonds(P, nL, n)
    got = kb.DimerMatrix(dpsi, bonds)
    nb = len(bonds)
    assert got["DD"].shape == (nb, nb) and got["D"].shape == (nb,) and got["flops"] > 0
    worst = 0.0
    for a in range(nb):
        worst = max(worst, abs(got["D"][a] - per_correlator_dimer(P, kb, dpsi, nL, n, bonds[a])))
        for b in range(nb):
            worst = max(worst, abs(got["DD"][a, b] - per_correlator_dimer(P, kb, dpsi, nL, n, bonds[a], bonds[b])))
    assert worst < 1e-12, worst


@pytest.mark.parametrize("qn", [0.0, 1.0])
def test_dimer_equals_the_spin_matrix_combination(P, ctx, orc, qn):
    """On truncated blocks <D_a> = SzSz + ½(SpSm + SmSp) at [i][j] of the spin correlation matrix, in either bond order."""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 6)
    kb = P.KronBlocks(pL, pR, [qn])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 5)
    n = 14
    nn, nnn = lattice_pairs(P, J1J2_CYL, n)
    bonds = nn + [p[::-1] for p in nnn] + [(0, n - 1), (n - 1, 0)]
    got = kb.DimerMatrix(dpsi, bonds)
    cm = kb.CorrelationMatrix(dpsi)
    ref = np.array([cm["SzSz"][i, j] + 0.5 * (cm["SpSm"][i, j] + cm["SmSp"][i, j]) for i, j in bonds])
    assert np.abs(got["D"] - ref).max() < 1e-12
    assert np.array_equal(got["DD"], got["DD"].T)


def _check_exact(P, ctx, ham, weights):
    blk, terms = exact_halves(P, ctx, ham)
    kb = P.KronBlocks(blk, blk, [0.0])
    e0, psi, st = kb.KronSumConstruct(terms).EPSSolve(tol=1e-12)
    assert st["converged"]
    N = ham["Lx"] * ham["Ly"]
    nn, nnn = lattice_pairs(P, ham, N)
    extra = [(0, N - 1), (N - 2, 1), (2, N // 2 + 1)]
    bonds = nn + nnn + extra
    got = kb.DimerMatrix(psi, bonds)
    e_ed, gap, dd_ref, d_ref = exact_dimers(terms, N, bonds)
    assert gap > 1e-6 and abs(e0 - e_ed) < 1e-9 * abs(e_ed)
    assert np.abs(got["DD"] - dd_ref).max() < 1e-8, np.abs(got["DD"] - dd_ref).max()
    assert np.abs(got["D"] - d_ref).max() < 1e-8, np.abs(got["D"] - d_ref).max()
    w = np.array([weights[0]] * len(nn) + [weights[1]] * len(nnn))
    assert abs(w @ got["D"][:len(w)] - e0) <= 1e-10 * abs(e0)
    # spin 1/2: (S_i·S_j)² = 3/16 − ½ S_i·S_j
    assert np.abs(np.diag(got["DD"]) - (3.0 / 16 - 0.5 * got["D"])).max() < 1e-10


def test_exact_blocks_match_exact_diagonalisation_chain12(P, ctx):
    """Un-truncated 6-site halves of the 12-site open Heisenberg chain: all 11 bonds plus longer pairs equal scipy ED, the
    bonds sum to the ground-state energy and <D_a²> = 3/16 − ½<D_a>."""
    _check_exact(P, ctx, HEIS_CHAIN12, (1.0, 0.0))


@pytest.mark.gpu
def test_exact_blocks_match_exact_diagonalisation_j1j2_4x4(P, ctx):
    """Un-truncated 8-site halves of the 4x4 J1-J2 cylinder: E0 = Σ_NN <D_a> + 0.5 Σ_NNN <D_a>."""
    if P.kind != "cuda":
        pytest.skip("16-site ED against the CUDA library only")
    _check_exact(P, ctx, J1J2_CYL, (1.0, 0.5))


def test_errors(P, ctx, orc):
    """62: psi, a bond array or an output NULL; 63: no bonds, a site outside [0, n), i == j (bond index in the message);
    56: not exactly one sector; 73: a block without Sz_i / Sp_i at a site some bond uses (site in the message)."""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 8)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 2)
    with pytest.raises(P.DmrgxError) as e:
        kb.DimerMatrix(None, [(0, 1)])
    assert e.value.code == 62
    L = P.lib()
    si, sj = np.array([0], np.int64), np.array([1], np.int64)
    dd, d = np.zeros(1), np.zeros(1)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for args in ((None, p(sj), p(dd), p(d)), (p(si), None, p(dd), p(d)), (p(si), p(sj), None, p(d)), (p(si), p(sj), p(dd), None)):
        assert L.dmrgx_dimer_matrix(kb.h, dpsi.ptr, C.c_longlong(1), *args, None) == 62
    assert L.dmrgx_dimer_matrix(kb.h, dpsi.ptr, C.c_longlong(1), p(si), p(sj), p(dd), p(d), None) == 0
    with pytest.raises(P.DmrgxError) as e:
        kb.DimerMatrix(dpsi, [])
    assert e.value.code == 63
    for bad in ((0, 16), (-1, 3), (5, 5)):
        with pytest.raises(P.DmrgxError) as e:
            kb.DimerMatrix(dpsi, [(0, 1), (2, 3), bad])
        assert e.value.code == 63 and "bond 2" in str(e.value), str(e.value)
    for qns in ([], [0.0, 1.0]):
        k2 = P.KronBlocks(pL, pR, qns)
        with pytest.raises(P.DmrgxError) as e:
            k2.DimerMatrix(ctx.vec(k2.NumStates(), np.ones(k2.NumStates())), [(0, 1)])
        assert e.value.code == 56
    b = P.Block.Initialize(ctx, 2, [1.0, 0.0, -1.0], [1, 2, 1])
    empty = (np.zeros(5, np.int64), np.zeros(0, np.int64), np.zeros(0))
    b.set_operator(P.OpSz, 0, *empty)
    b.set_operator(P.OpSp, 0, *empty)
    k3 = P.KronBlocks(b, P.Block.SingleSite(ctx), [0.5])
    x3 = ctx.vec(k3.NumStates(), np.ones(k3.NumStates()))
    with pytest.raises(P.DmrgxError) as e:
        k3.DimerMatrix(x3, [(0, 2), (2, 1)])
    assert e.value.code == 73 and "site 1" in str(e.value)
    got = k3.DimerMatrix(x3, [(0, 2)])   # only the sites the bonds use need operators
    assert got["DD"].shape == (1, 1)


@pytest.mark.gpu
def test_two_calls_are_bitwise_equal(P, ctx):
    """fixed plans and a fixed Gram summation order: no run-to-run noise (4x4 J1-J2 exact halves, D = 12870)"""
    if P.kind != "cuda":
        pytest.skip("the CUDA kernels only")
    blk, _ = exact_halves(P, ctx, J1J2_CYL)
    kb = P.KronBlocks(blk, blk, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 9)
    nn, nnn = lattice_pairs(P, J1J2_CYL, 16)
    a, b = kb.DimerMatrix(dpsi, nn + nnn), kb.DimerMatrix(dpsi, nn + nnn)
    for k in ("DD", "D"):
        assert np.array_equal(a[k], b[k]), k


# ---- the driver ----------------------------------------------------------------------------------------------------------

# the 4x4 J1-J2 cylinder, and a 4x2 one whose rungs NeighborPairs lists twice (periodic y with Ly = 2)
DRIVER_RUNS = [DRIVER_RUN, (["-Lx", 4, "-Ly", 2, "-J1", 0.5, "-Jz1", 1, "-J2", 0.25, "-Jz2", 0.5], dict(J1J2_CYL, Ly=2))]


def check_records(recs, cms, docs, ham):
    corr = docs["Correlations"]
    assert len(recs) == len(corr["values"]) == len(cms) >= 2
    ref = nn_bonds(ham)
    for rec, cm in zip(recs, cms):
        assert rec["GlobIdx"] == cm["GlobIdx"] and rec["LoopIdx"] == cm["LoopIdx"]
        assert [tuple(b["sites"]) for b in rec["bonds"]] == [p for p, _, _ in ref]
        assert [b["orientation"] for b in rec["bonds"]] == [o for _, o, _ in ref]
        assert [tuple(b["origin"]) for b in rec["bonds"]] == [r for _, _, r in ref]
        sites = cm["sites"]
        for b in rec["bonds"]:
            assert b["coords"] == [sites[b["sites"][0]], sites[b["sites"][1]]]
        D, DD = np.array(rec["Dimer"]), np.array(rec["DimerDimer"])
        nb = len(ref)
        assert DD.shape == (nb, nb)
        M = {k: np.array(cm[k]) for k in ("SzSz", "SpSm", "SmSp")}
        comb = np.array([M["SzSz"][i, j] + 0.5 * (M["SpSm"][i, j] + M["SmSp"][i, j]) for (i, j), _, _ in ref])
        assert np.abs(D - comb).max() < 1e-12, np.abs(D - comb).max()
        conn = DD - np.outer(D, D)
        for o, key in (("x", "DimerStructureFactorX"), ("y", "DimerStructureFactorY")):
            idx = [a for a in range(nb) if ref[a][1] == o]
            r = np.array([ref[a][2] for a in idx], float)
            S = np.array(rec[key])
            assert S.shape == (ham["Lx"], ham["Ly"])
            for kx in range(ham["Lx"]):
                for ky in range(ham["Ly"]):
                    ph = r @ np.array([2 * np.pi * kx / ham["Lx"], 2 * np.pi * ky / ham["Ly"]])
                    s = np.sum(np.cos(ph[:, None] - ph[None, :]) * conn[np.ix_(idx, idx)]) / len(idx)
                    assert abs(S[kx][ky] - s) < 1e-12, (key, kx, ky, S[kx][ky], s)


def test_driver_writes_the_dimer_matrix_at_every_measurement(P, exe, tmp_path):
    """-do_dimer_matrix 1 (with -do_correlation_matrix 1): one record per Correlations.json row over the distinct nearest-neighbour
    bonds, <D_a> equal to the spin-matrix combination, both structure factors reproduced from the record; without the option
    there is no file and the other outputs are byte for byte those of the run with it."""
    mw, ms = DRIVER_M[P.kind]
    for k, (args, ham) in enumerate(DRIVER_RUNS):
        docs, _ = dc.run_driver(exe, tmp_path / ("with%d" % k), args, mw, ms, extra=["-do_dimer_matrix", "1", "-do_correlation_matrix", "1"])
        out = str(tmp_path / ("with%d" % k) / "data") + "/"
        recs = json.load(open(out + "DimerMatrix.json"))
        cms = json.load(open(out + "CorrelationMatrix.json"))
        check_records(recs, cms, docs, ham)
        dc.run_driver(exe, tmp_path / ("without%d" % k), args, mw, ms)
        out0 = str(tmp_path / ("without%d" % k) / "data") + "/"
        assert not os.path.exists(out0 + "DimerMatrix.json")
        for f in ("DMRGSteps", "EntanglementSpectra", "Correlations"):
            assert open(out + f + ".json", "rb").read() == open(out0 + f + ".json", "rb").read(), f
