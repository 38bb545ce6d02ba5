"""The real-space dynamical correlation matrix: the Lanczos overlaps of dmrgx_spectral_lanczos_overlaps
(KronBlocks.SpectralLanczos(..., overlaps=True)), the host helpers dynamical_correlation and time_correlation, the device kernel
behind them (dev::gram_rect, through the test-only shim tests/devcheck/devcheck_gram_rect.cpp) and the driver's -do_dynamical_correlations output.
Every check runs on the host emulation of the device layer and, under -m gpu, on the CUDA library."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import driver_common as dc_driver
from devcheck_common import LD, Backend, assert_bound, assert_guards, bits, guard_for, rng_for, sentinel, wrap
from measure_common import (DRIVER_M, DRIVER_RUN, HEIS_CHAIN12, J1J2_CYL, SM, SP, SZ, P, ctx, dense_shell, exact_diagonalisation,  # noqa: F401
                            exact_halves, exe, ham_terms, ngpus, oracle_blocks, random_psi, start_vectors, tridiag)

OPS = (SZ, SP, SM)


def mixed_moments(r, v, kmax, shift=0.0):
    """‖phi_v‖ Σ_t ov[v, t, s]·((T_v - shift)^k)_{t,0} for k < kmax: a kmax × n array"""
    n = r["overlaps"].shape[2]
    k = int(r["nsteps_done"][v])
    if k == 0:
        return np.zeros((kmax, n))
    T = tridiag(r["alpha"][v], r["beta"][v], k) - shift * np.eye(k)
    x = np.zeros(k); x[0] = 1.0
    out = []
    for _ in range(kmax):
        out.append(np.sqrt(r["norm2"][v]) * (r["overlaps"][v, :k].T @ x))
        x = T @ x
    return np.array(out)


# ---- the library ---------------------------------------------------------------------------------------------------------

def test_overlaps_leave_the_recurrence_unchanged(P, ctx, orc):
    """alpha, beta, norm2 and nsteps_done of the overlaps call are bitwise those of the plain call, for all three ops and
    coefficient rows that leave some sites unused (those panels are built only for the overlaps)"""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 6)
    n = 14
    terms = ham_terms(P, J1J2_CYL, n)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 23)
    coef = np.random.default_rng(8).standard_normal((5, n))
    coef[:, [2, 9]] = 0.0
    coef[4] = np.eye(n)[6]
    for op in OPS:
        sh = P.KronBlocks(pL, pR, [float(op)]).KronSumConstruct(terms)
        a = kb.SpectralLanczos(dpsi, sh, op, coef, 5)
        b = kb.SpectralLanczos(dpsi, sh, op, coef, 5, overlaps=True)
        assert b["overlaps"].shape == (5, 5, n) and "overlaps" not in a
        for k in ("alpha", "beta", "norm2", "nsteps_done"):
            assert np.array_equal(bits(a[k]), bits(b[k])), (op, k)
        assert b["flops"] > a["flops"]


@pytest.mark.parametrize("case", ["L=R", "L!=R", "spin1"])
def test_mixed_moments_under_truncation(P, ctx, orc, case):
    """Oracle warm-up blocks of the 4x4 J1-J2 cylinder, random coefficients, ops Sz / S+ / S-, six steps: for k < 6,
    ‖phi_v‖ Σ_t ov·(T^k)_{t0} equals <P_s| H^k |phi_v>, with P_s = O_s psi from the dense block operators and H of the target
    sector from its shell.  This uses only the three-term relation, so it holds to rounding on truncated blocks."""
    nL, nR, spin = {"L=R": (8, 8, 1), "L!=R": (8, 6, 1), "spin1": (8, 8, 2)}[case]
    pL, pR = oracle_blocks(orc, P, ctx, nL, nR, spin)
    n = nL + nR
    terms = ham_terms(P, J1J2_CYL, n)
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, psi = random_psi(ctx, kb.NumStates(), 31)
    coef = np.random.default_rng(6).standard_normal((3, n))
    for op in OPS:
        tk = P.KronBlocks(pL, pR, [float(op)])
        sh = tk.KronSumConstruct(terms)
        r = kb.SpectralLanczos(dpsi, sh, op, coef, 6, overlaps=True)
        Ps = start_vectors(kb, tk, psi, op, np.eye(n))
        phi = coef @ Ps
        H = dense_shell(sh, tk.NumStates())
        scale = np.abs(np.linalg.eigvalsh(0.5 * (H + H.T))).max()
        pn = np.linalg.norm(Ps, axis=1)
        for v in range(3):
            assert r["nsteps_done"][v] == 6
            assert not r["overlaps"][v, 6:].any()
            got = mixed_moments(r, v, 6)
            x = phi[v].copy()
            for k in range(6):
                ref = Ps @ x
                tol = 1e-10 * pn * np.linalg.norm(phi[v]) * scale ** k
                assert (np.abs(got[k] - ref) <= tol).all(), (op, v, k, np.abs(got[k] - ref).max(), tol.min())
                x = H @ x


def _check_exact(P, ctx, ham, nsteps, eta, taus):
    """site sources c (coef = I) on exact halves, all three ops, against scipy ED of the whole lattice"""
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
    # the product's psi and ED's agree up to a sign, which cancels in every <0| A† f(H) B |0>
    Hsh = H - e_ed * sp.identity(2 ** N)
    for op in OPS:
        sh = H0 if op == SZ else P.KronBlocks(blk, blk, [float(op)]).KronSumConstruct(terms)
        r8 = kb.SpectralLanczos(dpsi, sh, op, np.eye(N), 8, overlaps=True)
        r = kb.SpectralLanczos(dpsi, sh, op, np.eye(N), nsteps, overlaps=True)
        Phi = np.array([ops[(op, s)] @ psi for s in range(N)])          # rows O_s |0>
        pn = np.linalg.norm(Phi, axis=1)
        sec = np.nonzero(ndown == N // 2 - op)[0]
        w, U = np.linalg.eigh(H[sec][:, sec].toarray())
        scale = max(abs(w[0] - e_ed), abs(w[-1] - e_ed))
        # mixed moments <0| O_s† (H - E0)^k O_c |0>, k < 8
        X = Phi.T.copy()
        got = np.array([mixed_moments(r8, c, 8, shift=e0) for c in range(N)])   # c, k, s
        for k in range(8):
            ref = Phi @ X                                                   # s, c
            tol = 1e-8 * np.outer(pn, pn) * scale ** k + 1e-14
            assert (np.abs(got[:, k, :].T - ref) <= tol).all(), (op, k, np.abs(got[:, k, :].T - ref).max())
            X = Hsh @ X
        # resolvent and propagator against the eigendecomposition of the target sector
        A = U.T @ Phi[:, sec].T                                            # eigenbasis × sites
        z = np.array([0.3, 1.0, 2.0, 3.5]) + e_ed + 1j * eta
        G = P.dynamical_correlation(r, z)                                  # c, s, z
        Gref = np.einsum("ks,kc,zk->csz", A, A, 1.0 / (z[:, None] - w[None, :]))
        assert G.shape == (N, N, len(z))
        assert np.abs(G - Gref).max() <= 1e-8, (op, np.abs(G - Gref).max())
        assert np.abs(G - G.transpose(1, 0, 2)).max() <= 1e-8
        Gt = P.time_correlation(r, taus, e0)
        Gtref = np.einsum("ks,kc,tk->cst", A, A, np.exp(-1j * np.outer(taus, w - e_ed)))
        assert np.abs(Gt - Gtref).max() <= 1e-8, (op, np.abs(Gt - Gtref).max())
        assert np.abs(Gt - Gt.transpose(1, 0, 2)).max() <= 1e-8
        # τ = 0 is the equal-time matrix
        assert np.abs(Gt[:, :, 0] - (Phi @ Phi.T).T).max() <= 1e-12


def test_exact_blocks_match_exact_diagonalisation_chain12(P, ctx):
    """Exact 6-site halves of the 12-site open Heisenberg chain, every site a source, all three ops: the mixed moments
    <0| O_s† (H - E0)^k O_c |0> for k < 8 match scipy ED, and with 120 steps the resolvent matrix at ω = 0.3, 1, 2, 3.5 above E0
    with η = 0.5 and the propagator at τ = 0 … 20 match ED to 1e-8, the matrix being symmetric in (s, c) to 1e-8.  (At η = 0.1
    the resolvent near ω = 3.5, where the spectrum is dense, still misses by 1e-5 after 160 steps.)"""
    _check_exact(P, ctx, HEIS_CHAIN12, 120, 0.5, np.array([0.0, 0.5, 1.0, 2.0, 5.0, 10.0, 20.0]))


@pytest.mark.gpu
def test_exact_blocks_match_exact_diagonalisation_j1j2_4x4(P, ctx):
    """The same on the 4x4 J1-J2 cylinder (D = 12870) at η = 0.5 and τ <= 20: its wider, denser spectrum takes 200 steps (after
    160 the resolvent at ω = 3.5 is still 3e-9 off and the propagator at τ = 20 2e-7)."""
    if P.kind != "cuda":
        pytest.skip("16-site ED against the CUDA library only")
    _check_exact(P, ctx, J1J2_CYL, 200, 0.5, np.array([0.0, 0.5, 1.0, 2.0, 5.0, 10.0, 20.0]))


def test_equal_time_identities_against_the_correlation_matrix(P, ctx, orc):
    """√norm2[v]·ov[v, 0, s] = <O_s psi, phi_v> is the coef-weighted row of SzSz, SpSm or SmSp of CorrelationMatrix (ops Sz,
    S-, S+), and Σ_s coef[v, s]·ov[v, 0, s] = √norm2[v], for qn = 0 and qn = 1"""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 6)
    n = 14
    terms = ham_terms(P, J1J2_CYL, n)
    coef = np.random.default_rng(12).standard_normal((4, n))
    for qn in (0.0, 1.0):
        kb = P.KronBlocks(pL, pR, [qn])
        dpsi, _ = random_psi(ctx, kb.NumStates(), 5)
        cm = kb.CorrelationMatrix(dpsi)
        for op, key in ((SZ, "SzSz"), (SM, "SpSm"), (SP, "SmSp")):
            tk = P.KronBlocks(pL, pR, [qn + op])
            if tk.NumStates() == 0:
                continue
            r = kb.SpectralLanczos(dpsi, tk.KronSumConstruct(terms), op, coef, 3, overlaps=True)
            ov0 = r["overlaps"][:, 0, :]
            tol = 1e-12 * max(1.0, np.abs(cm[key]).max() * np.abs(coef).sum(1).max())
            assert np.abs(np.sqrt(r["norm2"])[:, None] * ov0 - coef @ cm[key].T).max() <= tol, (qn, op)
            assert np.abs((coef * ov0).sum(1) - np.sqrt(r["norm2"])).max() <= tol, (qn, op)


def test_helpers_match_numpy_on_a_synthetic_recurrence():
    """dynamical_correlation and time_correlation equal ‖phi‖ Σ_t ov[t, s]·[f(T)]_{t0} computed with numpy inv / scipy expm
    on a random tridiagonal T; a vector with 0 steps gives 0; a scalar z or τ drops the last axis"""
    import dmrgx_loader
    import scipy.linalg as sl
    P = dmrgx_loader.load_package()
    rng = np.random.default_rng(3)
    nsteps, n = 6, 4
    a, b = rng.standard_normal((2, nsteps)), np.abs(rng.standard_normal((2, nsteps)))
    b[:, 0] = 0
    ov = rng.standard_normal((2, nsteps, n))
    ov[0, 5:] = 0
    r = {"alpha": a, "beta": b, "norm2": np.array([2.0, 3.0]), "nsteps_done": np.array([5, 0]), "overlaps": ov}
    z = np.array([0.3 + 0.1j, -1.0 + 0.05j, 2.0 + 1j])
    taus, e0 = np.array([0.0, 0.7, 3.0]), -0.4
    G, Gt = P.dynamical_correlation(r, z), P.time_correlation(r, taus, e0)
    assert G.shape == Gt.shape == (2, n, 3) and not G[1].any() and not Gt[1].any()
    T = tridiag(a[0], b[0], 5)
    for i, zi in enumerate(z):
        ref = np.sqrt(2.0) * ov[0, :5].T @ np.linalg.inv(zi * np.eye(5) - T)[:, 0]
        assert np.abs(G[0, :, i] - ref).max() < 1e-12 * np.abs(ref).max()
    for i, t in enumerate(taus):
        ref = np.sqrt(2.0) * ov[0, :5].T @ sl.expm(-1j * t * (T - e0 * np.eye(5)))[:, 0]
        assert np.abs(Gt[0, :, i] - ref).max() < 1e-12 * np.abs(ref).max()
    assert np.abs(P.dynamical_correlation(r, z[1]) - G[..., 1]).max() < 1e-13 * np.abs(G).max()
    assert np.abs(P.time_correlation(r, taus[2], e0) - Gt[..., 2]).max() < 1e-13 * np.abs(Gt).max()


def test_errors(P, ctx, orc):
    """62: overlaps NULL (and the inherited psi / target NULL); 63: no step, a bad op; 73: a block without operators at a site
    no coefficient uses, which the overlaps still need"""
    pL, pR = oracle_blocks(orc, P, ctx, 8, 8)
    n = 16
    kb = P.KronBlocks(pL, pR, [0.0])
    dpsi, _ = random_psi(ctx, kb.NumStates(), 1)
    H = kb.KronSumConstruct(ham_terms(P, J1J2_CYL, n))
    c = np.ones((1, n))

    def code(f):
        with pytest.raises(P.DmrgxError) as e:
            f()
        return e.value.code, str(e.value)
    out = [np.zeros(2) for _ in range(3)] + [np.zeros(1, np.int64)]
    pp = [o.ctypes.data_as(C.c_void_p) for o in out]
    assert P.lib().dmrgx_spectral_lanczos_overlaps(kb.h, dpsi.ptr, H.h, SZ, C.c_longlong(1), c.ctypes.data_as(C.c_void_p), C.c_longlong(2),
                                                   *pp, None, None) == 62
    assert code(lambda: kb.SpectralLanczos(None, H, SZ, c, 2, overlaps=True))[0] == 62
    assert code(lambda: kb.SpectralLanczos(dpsi, None, SZ, c, 2, overlaps=True))[0] == 62
    assert code(lambda: kb.SpectralLanczos(dpsi, H, SZ, c, 0, overlaps=True))[0] == 63
    assert code(lambda: kb.SpectralLanczos(dpsi, H, 2, c, 2, overlaps=True))[0] == 63
    b = P.Block.Initialize(ctx, 2, [1.0, 0.0, -1.0], [1, 2, 1])
    empty = (np.zeros(5, np.int64), np.zeros(0, np.int64), np.zeros(0))
    b.set_operator(P.OpSz, 0, *empty)
    b.set_operator(P.OpSp, 0, *empty)
    b.set_operator(P.OpH, 0, *empty)
    site = P.Block.SingleSite(ctx)
    k3 = P.KronBlocks(b, site, [0.5])
    h3 = k3.KronSumConstruct([])
    x3 = ctx.vec(k3.NumStates(), np.ones(k3.NumStates()))
    only = np.array([[1.0, 0.0, 1.0]])
    assert k3.SpectralLanczos(x3, h3, SZ, only, 2)["norm2"].shape == (1,)
    cd, msg = code(lambda: k3.SpectralLanczos(x3, h3, SZ, only, 2, overlaps=True))
    assert cd == 73 and "site 1" in msg


@pytest.mark.gpu
def test_determinism(P, ctx):
    """two calls give the same overlaps bits, and every vector of a 144-vector call the same bits as a call with that vector
    alone (4x4 J1-J2 exact halves, D = 12870)"""
    if P.kind != "cuda":
        pytest.skip("the CUDA kernels only")
    blk, terms = exact_halves(P, ctx, J1J2_CYL)
    kb = P.KronBlocks(blk, blk, [0.0])
    H = kb.KronSumConstruct(terms)
    dpsi, _ = random_psi(ctx, kb.NumStates(), 9)
    coef = np.random.default_rng(4).standard_normal((144, 16))
    a, b = kb.SpectralLanczos(dpsi, H, SZ, coef, 12, overlaps=True), kb.SpectralLanczos(dpsi, H, SZ, coef, 12, overlaps=True)
    for k in ("alpha", "beta", "norm2", "nsteps_done", "overlaps"):
        assert np.array_equal(bits(a[k]), bits(b[k])), k
    for v in range(144):
        one = kb.SpectralLanczos(dpsi, H, SZ, coef[v:v + 1], 12, overlaps=True)
        for k in ("alpha", "beta", "norm2", "nsteps_done", "overlaps"):
            assert np.array_equal(bits(one[k][0]), bits(a[k][v])), (k, v)


# ---- dev::gram_rect ------------------------------------------------------------------------------------------------------

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "dmrg.x_b200", "csrc")


@pytest.fixture(scope="module", params=["host", pytest.param("cuda", marks=pytest.mark.gpu)])
def dc(request):
    """the gram_rect shim over the host emulation or over the product's sm_100a object (conventions of test_device_kernels.py)"""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "devcheck", "libdevcheck_gram_rect_%s.so" % request.param)
    if not os.path.exists(path):
        subprocess.check_call(["make", "-s", "-C", CSRC, "devcheck-gram-rect-" + request.param])
    return Backend(request.param, path)


def gram_rect_call(dc, Pm, ldp, Qm, ldq, n, gs, gc, shift=0):
    np_, nq = len(Pm), len(Qm)
    g = guard_for(max(ldp, ldq))
    Pf, Qf = wrap(Pm, g), wrap(Qm, g)
    nG = (np_ - 1) * gs + (nq - 1) * gc + 1
    Gf = sentinel(nG, g)
    dc.ok("dc_gram_rect", Pf, Pf.size, ldp, np_, Qf, Qf.size, ldq, nq, n, shift, Gf, Gf.size, gs, gc, g)
    assert_guards(Gf, g, "G")
    G = Gf[g:-g]
    idx = np.arange(np_)[:, None] * gs + np.arange(nq)[None, :] * gc
    gap = np.ones(nG, bool)
    gap[idx.ravel()] = False
    assert (bits(G[gap]) == np.uint64(0xC3D5A5A55A5A0F0F)).all(), "a gap between strided elements was written"
    return G[idx]


def col_panel(rng, ncol, n, ld):
    M = np.full((ncol, ld), np.nan)
    M[:, :n] = rng.standard_normal((ncol, n))
    return M


@pytest.mark.parametrize("n", [8191, 8192, 8193])
def test_gram_rect_tiles_slabs_and_independence(dc, n):
    """np, nq in {1, 31, 32, 33, 72} across the 8192-row slab edge, with row-major, column-major and gapped strides: every
    element within the extended-precision summation bound of PᵀQ, and G[i][j] bitwise equal to the call with nq = 1 on column j
    (and np = 1 on row i) — an element's bits do not depend on the panel widths or on the tile that holds it"""
    rng = rng_for("gram_rect", n)
    ldp, ldq = (n + 4) & ~1, (n + 2) & ~1
    Pall, Qall = col_panel(rng, 72, n, ldp), col_panel(rng, 72, n, ldq)
    singles = {}
    for np_ in (1, 31, 32, 33, 72):
        for nq in (1, 31, 32, 33, 72):
            Pm, Qm = Pall[:np_], Qall[72 - nq:]
            gs, gc = [(nq, 1), (1, np_ + 3), (nq + 2, 1)][(np_ + nq) % 3]
            G = gram_rect_call(dc, Pm, ldp, Qm, ldq, n, gs, gc)
            A, B = Pm[:, :n].astype(LD), Qm[:, :n].astype(LD)
            assert_bound(G, A @ B.T, np.abs(A) @ np.abs(B).T, n, "gram_rect %dx%d n=%d" % (np_, nq, n))
            for j in sorted({0, nq // 2, nq - 1}):
                key = ("q", 72 - nq + j)
                if key not in singles:
                    singles[key] = gram_rect_call(dc, Pall, ldp, Qm[j:j + 1], ldq, n, 1, 1)[:, 0]
                assert (bits(G[:, j]) == bits(singles[key][:np_])).all(), (np_, nq, j)
            i = np_ - 1
            row = gram_rect_call(dc, Pm[i:i + 1], ldp, Qm, ldq, n, 1, 1)[0]
            assert (bits(G[i]) == bits(row)).all(), (np_, nq, i)
    assert (bits(gram_rect_call(dc, Pall, ldp, Qall, ldq, n, 72, 1)) == bits(gram_rect_call(dc, Pall, ldp, Qall, ldq, n, 72, 1))).all()


def test_gram_rect_every_column_alone_and_empty_rows(dc):
    """every column of a 72 × 72 call (n = 8193, two slabs) equals the nq = 1 call bit for bit; n = 0 writes zeros"""
    rng = rng_for("gram_rect-cols")
    n, ld = 8193, 8194
    Pm, Qm = col_panel(rng, 72, n, ld), col_panel(rng, 72, n, ld)
    G = gram_rect_call(dc, Pm, ld, Qm, ld, n, 72, 1)
    for j in range(72):
        assert (bits(G[:, j]) == bits(gram_rect_call(dc, Pm, ld, Qm[j:j + 1], ld, n, 1, 1)[:, 0])).all(), j
    Z = gram_rect_call(dc, Pm[:33], ld, Qm[:5], ld, 0, 5, 1)
    assert (bits(Z) == 0).all()


def test_gram_rect_refuses_misaligned_columns(dc):
    rng = rng_for("gram_rect-align")
    g = guard_for(12)
    Gf = sentinel(9, g)
    Pm = col_panel(rng, 3, 10, 12)
    Pf = wrap(np.concatenate([Pm.ravel(), [0.0]]), g)
    assert "16-byte" in dc.refused("dc_gram_rect", Pf, Pf.size, 12, 3, Pf, Pf.size, 12, 3, 10, 1, Gf, Gf.size, 3, 1, g)
    P11 = wrap(col_panel(rng, 3, 10, 11), g)
    P12 = wrap(Pm, g)
    assert "16-byte" in dc.refused("dc_gram_rect", P11, P11.size, 11, 3, P12, P12.size, 12, 3, 10, 0, Gf, Gf.size, 3, 1, g)
    assert "16-byte" in dc.refused("dc_gram_rect", P12, P12.size, 12, 3, P11, P11.size, 11, 3, 10, 0, Gf, Gf.size, 3, 1, g)


# ---- the driver ----------------------------------------------------------------------------------------------------------

def test_driver_writes_the_dynamical_correlations(P, exe, tmp_path):
    """-do_dynamical_correlations 1 with -do_spectral_function 1 -do_correlation_matrix 1 -spectral_nsteps 12: one record per
    measurement step aligned with the other two files; √norm2·overlaps[0] is the column of SzSz / SpSm / SmSp; the q-combined
    mixed moments (1/N) Σ_sc cos(q·(r_s - r_c)) M_k[s][c] equal the cos + sin moments of SpectralFunction.json; -dynamical_sources
    5,6 writes only those sources; a bad list is rejected; without the option no file."""
    mw, ms = DRIVER_M[P.kind]
    args, ham = DRIVER_RUN
    dc_driver.run_driver(exe, tmp_path / "with", args, mw, ms,
                         extra=["-do_dynamical_correlations", "1", "-do_spectral_function", "1", "-do_correlation_matrix", "1", "-spectral_nsteps", "12"])
    out = str(tmp_path / "with" / "data") + "/"
    recs = json.load(open(out + "DynamicalCorrelations.json"))
    sfs = json.load(open(out + "SpectralFunction.json"))
    cms = json.load(open(out + "CorrelationMatrix.json"))
    assert len(recs) == len(sfs) == len(cms) >= 2
    keys = {"zz": "SzSz", "pm": "SpSm", "mp": "SmSp"}
    for rec, sf, cm in zip(recs, sfs, cms):
        N = len(rec["sites"])
        assert rec["GlobIdx"] == sf["GlobIdx"] == cm["GlobIdx"] and rec["LoopIdx"] == sf["LoopIdx"] and rec["NSteps"] == 12
        assert rec["sites"] == cm["sites"] and rec["E0"] == sf["E0"] and rec["sources"] == list(range(N))
        r_xy = np.array(rec["sites"], float)
        for o, key in keys.items():
            ents = rec[o]
            assert [e["site"] for e in ents] == list(range(N))
            C = np.array(cm[key])
            M = np.zeros((12, N, N))                                 # k, s, c
            for c, e in enumerate(ents):
                k = e["steps"]
                assert len(e["alpha"]) == len(e["beta"]) == len(e["overlaps"]) == k <= 12 and (k == 0) == (e["norm2"] == 0)
                if k == 0:
                    continue
                ov = np.array(e["overlaps"])
                assert ov.shape == (k, N)
                assert np.abs(np.sqrt(e["norm2"]) * ov[0] - C[:, c]).max() <= 1e-10 * max(1.0, np.abs(C).max())
                T = tridiag(np.array(e["alpha"]), np.array(e["beta"]), k) - rec["E0"] * np.eye(k)
                x = np.zeros(k); x[0] = 1.0
                for kk in range(12):
                    M[kk, :, c] = np.sqrt(e["norm2"]) * ov.T @ x
                    x = T @ x
            scale = max(1.0, max(abs(a - rec["E0"]) + 2 * max(e["beta"] or [0]) for e in ents for a in e["alpha"] or [rec["E0"]]))
            for kx in range(ham["Lx"]):
                for ky in range(ham["Ly"]):
                    q = np.array([2 * np.pi * kx / ham["Lx"], 2 * np.pi * ky / ham["Ly"]])
                    ph = r_xy @ q
                    W = np.cos(ph[:, None] - ph[None, :]) / N
                    for kk in range(12):
                        ref = 0.0
                        for part in ("cos", "sin"):
                            p = sf[o][kx][ky][part]
                            if p["steps"] == 0:
                                continue
                            T = tridiag(np.array(p["alpha"]), np.array(p["beta"]), p["steps"]) - rec["E0"] * np.eye(p["steps"])
                            ref += p["norm2"] * np.linalg.matrix_power(T, kk)[0, 0]
                        got = float((W * M[kk]).sum())
                        assert abs(got - ref) <= 1e-9 * scale ** kk * max(1.0, np.abs(C).max() * N), (o, kx, ky, kk, got, ref)
    dc_driver.run_driver(exe, tmp_path / "two", args, mw, ms,
                         extra=["-do_dynamical_correlations", "1", "-dynamical_sources", "5,6", "-spectral_nsteps", "4", "-spectral_ops", "zz"])
    two = json.load(open(str(tmp_path / "two" / "data") + "/DynamicalCorrelations.json"))
    assert len(two) >= 2 and all(r["sources"] == [5, 6] and [e["site"] for e in r["zz"]] == [5, 6] and "pm" not in r for r in two)
    for bad, msg in (("5,5", "site 5 is listed twice"), ("3,16", "'16' is not a site index in [0, 16)"), ("x", "'x' is not a site index"),
                     (",", "the list is empty")):
        r = subprocess.run([exe] + [str(a) for a in args] + ["-mwarmup", "8", "-data_dir", str(tmp_path / "bad") + "/", "-do_dynamical_correlations", "1",
                                                             "-dynamical_sources", bad], capture_output=True, text=True, timeout=600)
        assert r.returncode != 0 and "-dynamical_sources: " + msg in r.stderr, (bad, r.stderr[-500:])
    dc_driver.run_driver(exe, tmp_path / "without", args, mw, ms, extra=["-do_spectral_function", "1", "-spectral_nsteps", "2"])
    assert not os.path.exists(str(tmp_path / "without" / "data") + "/DynamicalCorrelations.json")


@pytest.mark.gpu
@pytest.mark.skipif(ngpus() < 2, reason="needs two GPUs")
def test_two_rank_driver_rejects_the_option(P, exe, tmp_path):
    if P.kind != "cuda":
        pytest.skip("the CUDA executable only")
    args, _ = DRIVER_RUN
    cmd = [sys.executable, "-m", "torch.distributed.run", "--no-python", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", exe] + [str(a) for a in args] + ["-mwarmup", "16", "-do_dynamical_correlations", "1", "-data_dir", str(tmp_path) + "/"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode != 0 and "-do_dynamical_correlations runs on one GPU only" in r.stdout + r.stderr
