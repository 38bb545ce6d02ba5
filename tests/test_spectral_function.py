"""The continued-fraction recurrence of the dynamical structure factor (dmrgx_spectral_lanczos, KronBlocks.SpectralLanczos,
continued_fraction) and the driver's -do_spectral_function output.  Every check runs on the host emulation of the device layer
(tests/plancheck) and, under -m gpu, on the CUDA library."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import driver_common as dc
from measure_common import (DRIVER_M, DRIVER_RUN, HEIS_CHAIN12, J1J2_CYL, SM, SP, SZ, P, ctx, dense_shell,  # noqa: F401
                            exact_diagonalisation, exact_halves, exe, ham_terms, ngpus, oracle_blocks, random_psi,
                            start_vectors, tridiag)


# ---- references --------------------------------------------------------------------------------------------------------

def lanczos_moments(r, v, kmax, shift=0.0):
    k = int(r["nsteps_done"][v])
    if k == 0:
        return np.zeros(kmax)
    T = tridiag(r["alpha"][v], r["beta"][v], k) - shift * np.eye(k)
    x = np.zeros(k); x[0] = 1.0
    mu = []
    for _ in range(kmax):
        mu.append(r["norm2"][v] * x[0])
        x = T @ x
    return np.array(mu)


# ---- the library ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", ["L=R", "L!=R", "spin1"])
def test_moments_under_truncation(P, ctx, orc, case):
    """Oracle warm-up blocks of the 4x4 J1-J2 cylinder, random coefficients, ops Sz / S+ / S-, four steps: norm2·(T^k)_00 equals
    <phi| H^k |phi> for k < 8, with phi from the dense block operators and H of the target sector from its shell."""
    nL, nR, spin = {"L=R": (8, 8, 1), "L!=R": (8, 6, 1), "spin1": (8, 8, 2)}[case]
    pL, pR = oracle_blocks(orc, P, ctx, nL, nR, spin)
    terms = ham_terms(P, J1J2_CYL, nL + nR)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, psi = random_psi(ctx, kb.NumStates(), 17)
    coef = np.random.default_rng(5).standard_normal((3, nL + nR))
    for op in (SZ, SP, SM):
        tk = P.KronBlocks(pL, pR, [float(op)])
        sh = tk.KronSumConstruct(terms)
        r = kb.SpectralLanczos(dpsi, sh, op, coef, 4)
        assert r["alpha"].shape == (3, 4) and r["flops"] > 0 and not r["beta"][:, 0].any()
        phi = start_vectors(kb, tk, psi, op, coef)
        H = dense_shell(sh, tk.NumStates())
        scale = np.abs(np.linalg.eigvalsh(0.5 * (H + H.T))).max()
        for v in range(3):
            assert r["nsteps_done"][v] == 4
            ref, x = [], phi[v].copy()
            for k in range(8):
                ref.append(phi[v] @ x)
                x = H @ x
            got = lanczos_moments(r, v, 8)
            for k in range(8):
                assert abs(got[k] - ref[k]) <= 1e-10 * ref[0] * scale ** k, (op, v, k, got[k], ref[k])


def chain_coefs(N):
    """cos and sin of every chain momentum q = 2πk/N over the sites, /√N: rows 2k and 2k + 1"""
    c = []
    for k in range(N):
        ph = 2 * np.pi * k / N * np.arange(N)
        c += [np.cos(ph) / np.sqrt(N), np.sin(ph) / np.sqrt(N)]
    return np.array(c)


def _check_exact(P, ctx, ham, pole_steps):
    import scipy.sparse as sp
    N = ham["Lx"] * ham["Ly"]
    blk, terms = exact_halves(P, ctx, ham)
    kb = P.KronBlocks(blk, blk, [0.0])
    H0 = kb.KronSumConstruct(terms)
    e0, dpsi, st = H0.EPSSolve(tol=1e-12)
    assert st["converged"]
    w0, psi, H, ops, ndown = exact_diagonalisation(terms, N)
    e_ed = w0[0]
    assert abs(e0 - e_ed) < 1e-9 * abs(e_ed)
    coef = chain_coefs(N) if ham["Ly"] == 1 else None
    if coef is None:
        x = np.array([[s // ham["Ly"], s % ham["Ly"]] for s in range(N)], float)  # a momentum grid on the cylinder
        coef = []
        for kx in range(ham["Lx"]):
            for ky in range(ham["Ly"]):
                ph = x @ np.array([2 * np.pi * kx / ham["Lx"], 2 * np.pi * ky / ham["Ly"]])
                coef += [np.cos(ph) / np.sqrt(N), np.sin(ph) / np.sqrt(N)]
        coef = np.array(coef)
    for op in (SZ, SP, SM):
        tk = P.KronBlocks(blk, blk, [float(op)])
        sh = H0 if op == SZ else tk.KronSumConstruct(terms)
        r4 = kb.SpectralLanczos(dpsi, sh, op, coef, 4)
        rp = kb.SpectralLanczos(dpsi, sh, op, coef, pole_steps)
        sec = np.nonzero(ndown == N // 2 - op)[0]
        Hs = H[sec][:, sec].toarray()
        w, U = np.linalg.eigh(Hs)
        Hsh = H - e_ed * sp.identity(2 ** N)
        for v in range(len(coef)):
            phi = sum(coef[v, s] * (ops[(op, s)] @ psi) for s in range(N))
            ref, x = [], phi.copy()
            for k in range(8):
                ref.append(phi @ x)
                x = Hsh @ x
            scale = max(abs(w[0] - e_ed), abs(w[-1] - e_ed))
            got = lanczos_moments(r4, v, 8, shift=e0)
            for k in range(8):
                assert abs(got[k] - ref[k]) <= 1e-8 * max(ref[0], 1e-30) * scale ** k + 1e-14, (op, v, k, got[k], ref[k])
            if ref[0] < 1e-20:   # no weight (q = 0 of Sz, the sin part at q = 0 or π): nothing to locate
                continue
            # the lowest pole with non-negligible weight is the lowest excitation A_q reaches
            wt = (U.T @ phi[sec]) ** 2 / ref[0]
            n_ed = np.nonzero(wt > 1e-6)[0][0]
            k = int(rp["nsteps_done"][v])
            th, Y = np.linalg.eigh(tridiag(rp["alpha"][v], rp["beta"][v], k))
            j = np.nonzero(Y[0] ** 2 > 1e-6)[0][0]
            assert abs(th[j] - w[n_ed]) <= 1e-8 * max(1.0, abs(w[n_ed])), (op, v, th[j], w[n_ed])


def test_exact_blocks_match_exact_diagonalisation_chain12(P, ctx):
    """Exact 6-site halves of the 12-site open Heisenberg chain, every chain momentum and all three ops: the moments
    <0| A† (H - E0)^k A |0> match scipy ED, and after 40 steps the lowest pole with weight is the lowest excitation A_q reaches."""
    _check_exact(P, ctx, HEIS_CHAIN12, 40)


@pytest.mark.gpu
def test_exact_blocks_match_exact_diagonalisation_j1j2_4x4(P, ctx):
    if P.kind != "cuda":
        pytest.skip("16-site ED against the CUDA library only")
    # the frustrated 16-site spectrum is denser than the chain's: 40 steps leave the lowest pole of some A_q 1e-5 away, 80
    # converge every one to rounding
    _check_exact(P, ctx, J1J2_CYL, 80)


def test_sum_rules_against_the_correlation_matrix(P, ctx, orc):
    """norm2 = c·SzSz·c, c·SpSm·c, c·SmSp·c of CorrelationMatrix (ops Sz / S- / S+); with c = 1 and op Sz, phi = qn·psi: one
    step with α_0 = E0 for qn = 1, and norm2 = 0 with no step for qn = 0."""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 6)
    n = 14
    terms = ham_terms(P, J1J2_CYL, n)
    coef = np.random.default_rng(11).standard_normal((4, n))
    for qn in (0.0, 1.0):
        kb = P.KronBlocks(pL, pR, [qn])
        dpsi, _ = random_psi(ctx, kb.NumStates(), 3)
        cm = kb.CorrelationMatrix(dpsi)
        for op, key in ((SZ, "SzSz"), (SM, "SpSm"), (SP, "SmSp")):
            sh = kb.KronSumConstruct(terms) if op == SZ else P.KronBlocks(pL, pR, [qn + op]).KronSumConstruct(terms)
            r = kb.SpectralLanczos(dpsi, sh, op, coef, 3)
            ref = np.einsum("vi,ij,vj->v", coef, cm[key], coef)
            assert np.abs(r["norm2"] - ref).max() <= 1e-12 * max(1.0, np.abs(cm[key]).max() * np.abs(coef).sum(1).max() ** 2)
        H = kb.KronSumConstruct(terms)
        e0, gs, st = H.EPSSolve(tol=1e-12)
        r = kb.SpectralLanczos(gs, H, SZ, np.ones((1, n)), 5)
        if qn == 0.0:
            assert r["norm2"][0] == 0.0 and r["nsteps_done"][0] == 0 and not r["alpha"].any()
        else:
            assert r["nsteps_done"][0] == 1 and abs(r["norm2"][0] - qn * qn) < 1e-10
            assert abs(r["alpha"][0, 0] - e0) <= 1e-10 * abs(e0) and not r["alpha"][0, 1:].any() and not r["beta"].any()


def test_continued_fraction():
    """G(z) of a tridiagonal T equals norm2·((z - T)^-1)_00, for a batch and a vector of z; nsteps_done = 0 gives 0"""
    import dmrgx_loader
    P = dmrgx_loader.load_package()
    rng = np.random.default_rng(2)
    a, b = rng.standard_normal((2, 5)), np.abs(rng.standard_normal((2, 5)))
    b[:, 0] = 0
    z = np.array([0.3 + 0.1j, -1.0 + 0.05j, 2.0 + 1j])
    G = P.continued_fraction(a, b, [2.0, 3.0], [5, 0], z)
    assert G.shape == (2, 3) and not G[1].any()
    for i, zi in enumerate(z):
        ref = 2.0 * np.linalg.inv(zi * np.eye(5) - tridiag(a[0], b[0], 5))[0, 0]
        assert abs(G[0, i] - ref) < 1e-12 * abs(ref)
        assert abs(P.continued_fraction(a[0], b[0], 2.0, 3, zi) - 2.0 * np.linalg.inv(zi * np.eye(3) - tridiag(a[0], b[0], 3))[0, 0]) < 1e-12


def test_errors(P, ctx, orc):
    """62: psi, target or coef NULL; 63: bad op, no vector, no step, a non-finite coefficient; 56: not exactly one sector;
    73: a target of another sector or other blocks, a block without Sz / Sp at a site with a non-zero coefficient."""
    import ctypes as C
    pL, pR = oracle_blocks(orc, P, ctx, 8, 8)
    n = 16
    terms = ham_terms(P, J1J2_CYL, n)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 1)
    H = kb.KronSumConstruct(terms)
    c = np.ones((1, n))

    def code(f):
        with pytest.raises(P.DmrgxError) as e:
            f()
        return e.value.code, str(e.value)
    assert code(lambda: kb.SpectralLanczos(None, H, SZ, c, 2))[0] == 62
    assert code(lambda: kb.SpectralLanczos(dpsi, None, SZ, c, 2))[0] == 62
    out = [np.zeros(2) for _ in range(3)] + [np.zeros(1, np.int64)]
    pp = [o.ctypes.data_as(C.c_void_p) for o in out]
    assert P.lib().dmrgx_spectral_lanczos(kb.h, dpsi.ptr, H.h, SZ, C.c_longlong(1), None, C.c_longlong(2), *pp, None) == 62
    assert P.lib().dmrgx_spectral_lanczos(kb.h, dpsi.ptr, H.h, SZ, C.c_longlong(1), c.ctypes.data_as(C.c_void_p), C.c_longlong(2), pp[0], None,
                                          pp[2], pp[3], None) == 62
    assert code(lambda: kb.SpectralLanczos(dpsi, H, 2, c, 2))[0] == 63
    assert code(lambda: kb.SpectralLanczos(dpsi, H, SZ, np.zeros((0, n)), 2))[0] == 63
    assert code(lambda: kb.SpectralLanczos(dpsi, H, SZ, c, 0))[0] == 63
    bad = c.copy(); bad[0, 3] = np.nan
    assert code(lambda: kb.SpectralLanczos(dpsi, H, SZ, bad, 2))[0] == 63
    for qns in ([], [0.0, 1.0]):
        k2 = P.KronBlocks(pL, pR, qns)
        assert code(lambda: k2.SpectralLanczos(ctx.vec(k2.NumStates(), np.ones(k2.NumStates())), H, SZ, c, 2))[0] == 56
    hp = P.KronBlocks(pL, pR, [1.0]).KronSumConstruct(terms)
    assert code(lambda: kb.SpectralLanczos(dpsi, hp, SZ, c, 2))[0] == 73      # sector qn + 1 for op Sz
    assert code(lambda: kb.SpectralLanczos(dpsi, H, SP, c, 2))[0] == 73       # sector qn for op S+
    q6, _ = oracle_blocks(orc, P, ctx, 8, 6)
    other = P.KronBlocks(q6, pR, [0.0])
    assert code(lambda: kb.SpectralLanczos(dpsi, other.KronSumConstruct(ham_terms(P, J1J2_CYL, 16)), SZ, c, 2))[0] == 73
    b = P.Block.Initialize(ctx, 2, [1.0, 0.0, -1.0], [1, 2, 1])
    empty = (np.zeros(5, np.int64), np.zeros(0, np.int64), np.zeros(0))
    b.set_operator(P.OpSz, 0, *empty)
    b.set_operator(P.OpSp, 0, *empty)
    b.set_operator(P.OpH, 0, *empty)
    site = P.Block.SingleSite(ctx)
    k3 = P.KronBlocks(b, site, [0.5])
    h3 = k3.KronSumConstruct([])
    x3 = ctx.vec(k3.NumStates(), np.ones(k3.NumStates()))
    cd, msg = code(lambda: k3.SpectralLanczos(x3, h3, SZ, np.ones((1, 3)), 2))
    assert cd == 73 and "site 1" in msg
    r = k3.SpectralLanczos(x3, h3, SZ, np.array([[1.0, 0.0, 1.0]]), 2)   # only the sites with a coefficient need operators
    assert r["norm2"].shape == (1,)


@pytest.mark.gpu
def test_determinism(P, ctx):
    """fixed per-column summation orders: two calls give the same bits, and every vector of a 144-vector call the same bits as
    a call with that vector alone (4x4 J1-J2 exact halves, D = 12870)"""
    if P.kind != "cuda":
        pytest.skip("the CUDA kernels only")
    blk, terms = exact_halves(P, ctx, J1J2_CYL)
    kb = P.KronBlocks(blk, blk, [0.0])
    H = kb.KronSumConstruct(terms)
    dpsi, _ = random_psi(ctx, kb.NumStates(), 9)
    coef = np.random.default_rng(4).standard_normal((144, 16))
    a, b = kb.SpectralLanczos(dpsi, H, SZ, coef, 12), kb.SpectralLanczos(dpsi, H, SZ, coef, 12)
    for k in ("alpha", "beta", "norm2", "nsteps_done"):
        assert np.array_equal(a[k], b[k]), k
    for v in range(144):
        one = kb.SpectralLanczos(dpsi, H, SZ, coef[v:v + 1], 12)
        for k in ("alpha", "beta", "norm2", "nsteps_done"):
            assert np.array_equal(one[k][0], a[k][v]), (k, v)


# ---- the driver ----------------------------------------------------------------------------------------------------------

def test_driver_writes_the_spectral_function(P, exe, tmp_path):
    """-do_spectral_function 1 (with -do_correlation_matrix 1): one record per Correlations.json row; summed over cos / sin,
    zz + (pm + mp)/2 of norm2 is the step's StructureFactor; a bad -spectral_ops is rejected; without the option no file."""
    mw, ms = DRIVER_M[P.kind]
    args, ham = DRIVER_RUN
    docs, _ = dc.run_driver(exe, tmp_path / "with", args, mw, ms,
                            extra=["-do_spectral_function", "1", "-do_correlation_matrix", "1", "-spectral_nsteps", "12"])
    out = str(tmp_path / "with" / "data") + "/"
    recs = json.load(open(out + "SpectralFunction.json"))
    cms = json.load(open(out + "CorrelationMatrix.json"))
    assert len(recs) == len(docs["Correlations"]["values"]) == len(cms) >= 2
    steps = {row[0]: row[-1] for row in docs["DMRGSteps"]["table"]}
    for rec, cm in zip(recs, cms):
        assert rec["GlobIdx"] == cm["GlobIdx"] and rec["LoopIdx"] == cm["LoopIdx"] and rec["NSteps"] == 12
        assert rec["sites"] == cm["sites"] and abs(rec["E0"] - steps[rec["GlobIdx"]]) <= 1e-10 * abs(rec["E0"])
        for kx in range(ham["Lx"]):
            for ky in range(ham["Ly"]):
                s = 0.0
                for part in ("cos", "sin"):
                    for o, w in (("zz", 1.0), ("pm", 0.5), ("mp", 0.5)):
                        e = rec[o][kx][ky][part]
                        assert len(e["alpha"]) == len(e["beta"]) == e["steps"] <= 12
                        assert (e["steps"] == 0) == (e["norm2"] == 0)
                        s += w * e["norm2"]
                assert abs(s - cm["StructureFactor"][kx][ky]) < 1e-10, (kx, ky, s, cm["StructureFactor"][kx][ky])
    r = subprocess.run([exe] + [str(a) for a in args] + ["-mwarmup", "8", "-data_dir", str(tmp_path / "bad") + "/", "-do_spectral_function", "1",
                                                         "-spectral_ops", "zz,xy"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "-spectral_ops: unknown item 'xy'" in r.stderr
    dc.run_driver(exe, tmp_path / "without", args, mw, ms)
    assert not os.path.exists(str(tmp_path / "without" / "data") + "/SpectralFunction.json")


@pytest.mark.gpu
@pytest.mark.skipif(ngpus() < 2, reason="needs two GPUs")
def test_two_rank_driver_rejects_the_option(P, exe, tmp_path):
    if P.kind != "cuda":
        pytest.skip("the CUDA executable only")
    args, _ = DRIVER_RUN
    cmd = [sys.executable, "-m", "torch.distributed.run", "--no-python", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", exe] + [str(a) for a in args] + ["-mwarmup", "16", "-do_spectral_function", "1", "-data_dir", str(tmp_path) + "/"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode != 0 and "one GPU only" in r.stdout + r.stderr
