"""Parity tests proper (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle on the same seeded
inputs, plus size-independent properties at larger sizes.  Tolerances: H·psi 1e-13 relative (per term), energies and
truncation errors 1e-10 relative (north_star), bookkeeping bit-exact."""
import os

import numpy as np

import libswitch
import pytest

import parity_common as pc
from devcheck_common import eig_inputs

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def P():
    import dmrgx_loader
    P = dmrgx_loader.load_package()
    libswitch.use_library(P, None)  # the real CUDA library, nothing else
    return P


@pytest.fixture(scope="module")
def ctx(P):
    c = P.Context(0)
    yield c
    c.close()


HEIS_CHAIN = dict(Lx=16, Ly=1, J1=0.5, Jz1=1.0, J2=0.0, Jz2=0.0, bcx=0, bcy=0)
J1J2_CYL = dict(Lx=4, Ly=4, J1=0.5, Jz1=1.0, J2=0.25, Jz2=0.5)
HEIS_CYL = dict(Lx=6, Ly=2, J1=0.5, Jz1=1.0, J2=0.0, Jz2=0.0)
XY_CYL = dict(Lx=4, Ly=4, J1=1.0, Jz1=0.0, J2=1.0, Jz2=0.0)


def test_native_library_is_loaded(P, ctx):
    assert os.path.realpath(P.lib()._name) == os.path.realpath(P.LIB_PATH)
    n0 = P.launch_count()
    v = ctx.vec(10, np.arange(10.0))
    assert v.get().tolist() == list(range(10))
    b = P.Block.SingleSite(ctx)
    assert b.NumStates() == 2
    assert P.launch_count() >= n0


def test_single_site_blocks(P, ctx, orc):
    for spin in (1, 2):
        pc.assert_blocks_equal(P, orc, P.Block.SingleSite(ctx, spin), orc.Block.single_site(spin), tol=0.0)


@pytest.mark.parametrize("ham,nsys,nenv,mprep,mkeep", [
    (HEIS_CHAIN, 3, 3, 8, 6),
    (HEIS_CHAIN, 5, 3, 16, 12),
    (HEIS_CHAIN, 7, 7, 24, 20),
    (HEIS_CYL, 4, 4, 12, 10),
    (J1J2_CYL, 5, 5, 20, 16),
    (J1J2_CYL, 7, 7, 40, 32),
    (XY_CYL, 7, 7, 32, 24),
], ids=["chain-3+3", "chain-5+3", "chain-7+7", "cyl6x2-4+4", "j1j2-5+5", "j1j2-7+7", "xy-7+7"])
def test_single_dmrg_step_matches_oracle(P, ctx, orc, ham, nsys, nenv, mprep, mkeep):
    rng = np.random.default_rng(7)
    pc.run_step_parity(P, orc, ctx, ham, nsys, nenv, mprep, mkeep, rng)


@pytest.mark.parametrize("config,m", [("j1j2_12x6", 64), ("j1j2_12x6", 160), ("heis_8x4", 96), ("heis_chain24", 64), ("xy_16x8", 80)])
def test_synthetic_workload_matvec_matches_oracle(P, ctx, orc, config, m):
    """BASELINE.json configs on synthetic truncated blocks (bench_workload.py) at sizes the oracle finishes in seconds."""
    import bench_workload as W
    wl = W.Workload(P, ctx, config, m=m)
    enl_o, kb_o = W.oracle_side(orc, wl)
    pc.assert_blocks_equal(P, orc, wl.enl, enl_o, what="enlarged synthetic block")
    pc.check_kron_bookkeeping(P, orc, wl.kron, kb_o)
    osh = orc.Shell(kb_o, wl.terms)
    pc.check_matvec(P, orc, ctx, wl.shell, osh, np.random.default_rng(3), nvec=2)


def _row_windows(kron, nrows):
    """>= 3 windows of superblock rows: across the start of the largest sector pair (ragged edge tile of the previous pair next
    to full tiles), in its middle (full 64x64 tiles, long stage-2 chains that the planner may split), across its end."""
    _, _, _, _, off = kron.data()
    sizes = np.diff(off)
    big = int(np.argmax(sizes))
    n = int(off[-1])
    h = nrows // 2
    a, e = int(off[big]), int(off[big + 1])
    mid = a + (e - a) // 2
    return [(max(0, c - h), min(n, c + h)) for c in (a, mid, e)] + [(0, min(n, nrows))]


@pytest.mark.parametrize("config,m,nrows", [("j1j2_12x6", 512, 2048), ("j1j2_12x6", 1024, 1024), ("j1j2_12x6", 2048, 384),
                                            ("heis_8x4", 768, 1024), ("xy_16x8", 640, 1024)])
def test_headline_tile_sizes_match_oracle_on_row_windows(P, ctx, orc, config, m, nrows):
    """The code that runs the flops of the metric's configuration — full 64x64 unit-coefficient DMMA tiles, cells tiled into
    several 64-wide items, K spanning many chunks, stage-2 chains split into parts + reduce_kernel — against the oracle's
    restatement of MatMult_KronSumShell (src/DMRGKron.cpp:1844-1864) on windows of rows: largest enlarged sector > 64 at
    m = 512 (~200), > 128 at m = 1024 (~400) and the metric's own m = 2048 (~800)."""
    import bench_workload as W
    import os as _os
    wl = W.Workload(P, ctx, config, m=m)
    q, s = wl.enl.sectors()
    assert s.max() > 128
    _, kb_o = W.oracle_side(orc, wl)
    pc.check_kron_bookkeeping(P, orc, wl.kron, kb_o)
    st = wl.shell.stats()
    x = wl.random_state(9)
    y = wl.shell.MatMult_host(x)
    scale = np.abs(y).max()
    cores = _os.cpu_count() or 1
    worst = 0.0
    for (r0, r1) in _row_windows(wl.kron, nrows):
        y_ref = orc.Shell(kb_o, wl.terms, rows=(r0, r1)).apply(x, cores)
        worst = max(worst, np.abs(y[r0:r1] - y_ref).max() / scale)
    assert worst <= pc.MATVEC_RTOL * st["nterms"], worst
    if m >= 2048:   # the planner did split stage-2 chains here (reduce_kernel in play)
        assert st["tiles_stage2"] > 1000


@pytest.mark.parametrize("m,keep", [(256, 200), (384, 300)])
def test_truncation_and_rotation_match_oracle_at_larger_sectors(P, ctx, orc, m, keep):
    """GetTruncation / RotateOperators with reduced-density-matrix blocks beyond the 64-state shared-memory solver (largest
    block ~100 at m = 256, ~150 at m = 384): both sides get the SAME psi (the product's converged ground state), so the
    kept-state counts, spectra and truncation errors are comparable bit for bit / to 1e-10."""
    import bench_workload as W
    wl = W.Workload(P, ctx, "heis_8x4", m=m)
    enl_o, kb_o = W.oracle_side(orc, wl)
    q, s = wl.enl.sectors()
    assert s.max() > 64
    e, psi, st = wl.shell.EPSSolve(tol=1e-11)
    assert st["converged"]
    ph = psi.get()
    for keep in range(keep, keep + 8):   # move the cut off a degenerate multiplet (the oracle reports ties)
        obtL = orc.Truncation(kb_o, ph, keep, True)
        obtR = orc.Truncation(kb_o, ph, keep, False)
        if not (obtL.tie or obtR.tie):
            break
    pbtL, pbtR = P.GetTruncation(wl.kron, psi, keep)
    pc.check_truncation(P, orc, pbtL, obtL, None)
    pc.check_truncation(P, orc, pbtR, obtR, None)
    pnew = P.RotateOperators(wl.enl, pbtL)
    Up = pbtL.RotMatT()
    HL = enl_o.get_op_dense(orc.OP_H)
    assert np.abs(pc.dense_op(pnew, P.OpH) - Up @ HL @ Up.T).max() < 1e-11 * max(1.0, np.abs(HL).max())
    for i in wl.used[:3] + [wl.nsites_blk]:
        for pop, oop in ((P.OpSp, orc.OP_SP), (P.OpSz, orc.OP_SZ)):
            O_enl = enl_o.get_op_dense(oop, i)
            assert np.abs(pc.dense_op(pnew, pop, i) - Up @ O_enl @ Up.T).max() < 1e-11
    assert pnew.CheckOperatorBlocks() == 0


@pytest.mark.parametrize("a_k,b_k", [(1, 1), (1, 0), (0, 1), (0, 0)])
def test_contraction_engine_selftest(P, ctx, a_k, b_k):
    """dmrgx_selftest_gemm: the chain kernel on plain products against a double-double-free host reference computed inside the
    library from the same seeded operands — all four operand layouts, full and ragged tiles (48 / 32 / 16 wide edges), one
    segment and a chain of 8."""
    import ctypes as C
    L = P.lib()
    for (M, N, K, nseg) in [(256, 320, 512, 1), (256, 320, 512, 8), (64 * 3 + 48, 64 * 2 + 32, 200, 1), (64 + 16, 64 * 2 + 48, 77, 3), (40, 24, 33, 2)]:
        ms, err = C.c_double(), C.c_double()
        rc = L.dmrgx_selftest_gemm(ctx.h, C.c_longlong(M), C.c_longlong(N), C.c_longlong(K), a_k, b_k, nseg, 1, C.byref(ms), C.byref(err))
        assert rc == 0, L.dmrgx_last_error()
        assert err.value <= 1e-13 * K * nseg, (M, N, K, nseg, err.value)


def _oracle_exact_chain(orc, nhalf):
    """the oracle's own exact halves of the open Heisenberg chain (same enlargement sequence as ExactChainWorkload)"""
    T = lambda n: orc.ham_terms(2 * nhalf, 1, 0.5, 1.0, 0.0, 0.0, n, 0, 0)
    site = orc.Block.single_site()
    blk = orc.Block.single_site()
    for n in range(2, nhalf + 1):
        blk = orc.kron_eye(blk, site, T(n))
    return blk, orc.KronBlocks(blk, blk, [0.0]), T(2 * nhalf)


@pytest.mark.parametrize("nhalf", [9, 12, 13])
def test_sparse_sector_kernel_matches_oracle_and_chain_kernel(P, ctx, orc, nhalf, monkeypatch):
    """spmm_kernel (the sparse-sector matvec of un-truncated blocks) against (a) the oracle's restatement of
    MatMult_KronSumShell on row windows and (b) the chain kernel's sparse segments on the whole vector (two independent
    kernels).  nhalf = 12 is the benchmark's workload (right sectors up to 924 wide: four column chunks per thread);
    nhalf = 13 has right sectors 1716 wide (two passes of the column super-chunk loop)."""
    import bench_workload as W
    sw = W.ExactChainWorkload(P, ctx, nhalf)
    st = sw.shell.stats()
    assert st["tiles_stage1"] == 0 and st["tiles_stage2"] > 0          # the sparse plan is in use
    l0 = P.launch_count()
    x = sw.random_state(3)
    y = sw.shell.MatMult_host(x)
    assert P.launch_count() - l0 == 1                                   # one launch per apply
    oblk, okb, terms = _oracle_exact_chain(orc, nhalf)
    pc.check_kron_bookkeeping(P, orc, sw.kron, okb)
    n = sw.n
    scale = np.abs(y).max()
    _, _, _, _, off = sw.kron.data()
    big = int(np.argmax(np.diff(off)))
    for c in (0, int(off[big]), int(off[big]) + int(np.diff(off)[big]) // 2, int(off[big + 1]), n):
        r0, r1 = max(0, c - 1500), min(n, c + 1500)
        y_ref = orc.Shell(okb, terms, rows=(r0, r1)).apply(x, 4)
        assert np.abs(y[r0:r1] - y_ref).max() <= 1e-13 * scale * 5
    monkeypatch.setenv("DMRGX_NO_SPARSE", "1")
    dense_path = sw.kron.KronSumConstruct(sw.terms)
    monkeypatch.delenv("DMRGX_NO_SPARSE")
    assert dense_path.stats()["tiles_stage2"] > 0 and dense_path.stats()["tiles_stage1"] > 0
    y2 = dense_path.MatMult_host(x)
    assert np.abs(y - y2).max() <= 1e-13 * scale * 5


@pytest.mark.parametrize("config,m", [("j1j2_12x6", 96), ("heis_8x4", 128), ("xy_16x8", 72)])
def test_sparse_sector_kernel_general_csr_factors(P, ctx, orc, config, m, monkeypatch):
    """the same kernel with BOTH factors of the L-R terms general CSR matrices and rows longer than one preload batch:
    sector-dense synthetic blocks uploaded with the dense threshold above 1, so every tile is stored as CSR."""
    import bench_workload as W
    wl = W.Workload(P, ctx, config, m=m)
    enl_o, kb_o = W.oracle_side(orc, wl)
    try:
        ctx.set_dense_threshold(2.0)
        up = pc.upload_block(P, ctx, enl_o, orc)      # the ENLARGED block handed over as CSR (route B of INTEGRATION.md)
    finally:
        ctx.set_dense_threshold(0.125)
    monkeypatch.setenv("DMRGX_FORCE_SPARSE", "1")   # these blocks are 100 % filled inside their sectors: skip the planner's fill criterion
    shell = P.KronBlocks(up, up, [0.0]).KronSumConstruct(wl.terms)
    monkeypatch.delenv("DMRGX_FORCE_SPARSE")
    st = shell.stats()
    assert st["tiles_stage1"] == 0 and st["tiles_stage2"] > 0          # the sparse plan is in use
    pc.check_matvec(P, orc, ctx, shell, orc.Shell(kb_o, wl.terms), np.random.default_rng(3), nvec=1)


def _eig_selftest(P, ctx, mats):
    import ctypes as C
    n = np.array([m.shape[0] for m in mats], np.int64)
    a = np.concatenate([np.ascontiguousarray(m).ravel() for m in mats])
    w = np.zeros(int(n.sum()))
    ms = C.c_double()
    rc = P.lib().dmrgx_selftest_eig(ctx.h, C.c_longlong(len(mats)), n.ctypes.data_as(C.c_void_p), a.ctypes.data_as(C.c_void_p), w.ctypes.data_as(C.c_void_p), C.byref(ms))
    assert rc == 0, P.lib().dmrgx_last_error()
    out, oa, ow = [], 0, 0
    for k in n:
        out.append((w[ow:ow + k], a[oa:oa + k * k].reshape(k, k)))
        oa += k * k; ow += k
    return out, ms.value


@pytest.mark.parametrize("case", [[65, 96, 128], [130, 200, 333, 64, 17, 1], [512, 700, 257], [832, 640, 448, 250, 120, 832, 640, 448, 250, 120],
                                  [1, 2, 63, 64, 65, 127, 128, 129, 192, 193], "multiplets", "diagonal", "zero", "indefinite", "negative-definite",
                                  "batch-300"],
                         ids=["just-above-64", "mixed", "medium", "m2048-like", "switch-and-padding-edges", "multiplets", "diagonal", "zero",
                              "indefinite", "negative-definite", "batch-300"])
def test_batched_block_jacobi_eigensolver(P, ctx, case):
    """The library's own eigensolver for reduced-density-matrix blocks (EigRDM_BlockDiag, include/DMRGBlockContainer.hpp:1962-2003;
    no cuSOLVER): rho-like matrices X·X^T with a fast-decaying spectrum (rank-deficient, eigenvalues down to round-off) at
    the sizes of the cyclic-Jacobi / block-Jacobi switch and of the 64-padding, exact multiplets, diagonal, zero,
    indefinite and negative-definite inputs and one batch of 300 small blocks, against numpy's LAPACK: eigenvalues to
    5e-14 of the norm, residual and orthogonality to 1e-13."""
    mats = eig_inputs(case)
    res, ms = _eig_selftest(P, ctx, mats)
    for (w, V), R in zip(res, mats):
        ref = np.linalg.eigvalsh(R)
        nrm = np.abs(ref).max()
        assert np.all(np.diff(w) >= 0)
        # LAPACK itself promises O(n·eps·||A||); the Rayleigh quotients carry the rounding of one n-term product
        assert np.abs(w - ref).max() <= 5e-14 * nrm + 1e-17
        assert np.abs(V @ V.T - np.eye(len(w))).max() <= 1e-12          # rows orthonormal
        assert np.abs(V @ R @ V.T - np.diag(w)).max() <= 2e-13 * nrm + 1e-17


def test_sparse_and_dense_tile_paths_agree(P, ctx, orc):
    rng = np.random.default_rng(11)
    ham = J1J2_CYL
    d = orc.DMRG(ham["Lx"], ham["Ly"], ham["J1"], ham["Jz1"], ham["J2"], ham["Jz2"])
    d.warmup(24)
    oL = orc.kron_eye(d.block(6), orc.Block.single_site(), pc.lr_terms(orc, ham, 8))
    okb = orc.KronBlocks(oL, oL, [0.0])
    terms = pc.lr_terms(orc, ham, 16)
    osh = orc.Shell(okb, terms)
    x = rng.standard_normal(osh.n)
    y_ref = osh.apply(x)
    try:
        for thr in (0.0, 2.0):
            ctx.set_dense_threshold(thr)
            pL = pc.upload_block(P, ctx, oL, orc)
            psh = P.KronBlocks(pL, pL, [0.0]).KronSumConstruct(terms)
            y = psh.MatMult_host(x)
            assert np.abs(y - y_ref).max() <= 1e-12 * np.abs(y_ref).max()
    finally:
        ctx.set_dense_threshold(0.125)


def test_full_size_properties_m2048(P, ctx):
    """BASELINE.json's full size (12x6, m=2048): no oracle can run here, so check size-independent properties of H·psi:
    linearity, symmetry <x|Hy> = <Hx|y>, and the Rayleigh quotient bound of the Lanczos result."""
    import bench_workload as W
    wl = W.Workload(P, ctx, "j1j2_12x6", m=2048)
    H = wl.shell
    n = wl.n
    assert n > 1_000_000
    rng = np.random.default_rng(0)
    x = rng.standard_normal(n); y = rng.standard_normal(n)
    Hx = H.MatMult_host(x); Hy = H.MatMult_host(y)
    Hxy = H.MatMult_host(2.0 * x - 3.0 * y)
    scale = max(np.abs(Hx).max(), np.abs(Hy).max())
    assert np.abs(Hxy - (2.0 * Hx - 3.0 * Hy)).max() <= 1e-11 * scale
    assert abs(y @ Hx - x @ Hy) <= 1e-10 * np.linalg.norm(Hx) * np.linalg.norm(y)
    e, psi, st = H.EPSSolve(tol=1e-6, max_it=3)
    p = psi.get()
    assert abs(np.linalg.norm(p) - 1.0) < 1e-10
    ray = p @ H.MatMult_host(p)
    assert abs(ray - e) <= 1e-8 * max(1.0, abs(e))
    assert e < (x @ Hx) / (x @ x)  # below a random vector's Rayleigh quotient


def test_truncate_rotate_roundtrip_properties(P, ctx):
    """Synthetic m=256 step: U rows orthonormal, kept weights + truncation error = 1, rotated H symmetric."""
    import bench_workload as W
    wl = W.Workload(P, ctx, "heis_8x4", m=256)
    e, psi, st = wl.shell.EPSSolve(tol=1e-10)
    assert st["converged"]
    btL, btR = P.GetTruncation(wl.kron, psi, 200)
    for bt in (btL, btR):
        U = bt.RotMatT()
        assert np.abs(U @ U.T - np.eye(bt.m)).max() < 1e-10
        ev, _ = bt.spectrum()
        assert abs(ev.sum() - 1.0) < 1e-10
        kept = np.sort(ev)[::-1][:bt.m]
        assert abs((1.0 - kept[kept > 0].sum()) - bt.TruncErr) < 1e-12
    new = P.RotateOperators(wl.enl, btL)
    assert new.NumStates() == btL.m and new.CheckOperatorBlocks() == 0
    Hn = new.get_operator_dense(P.OpH)
    assert np.abs(Hn - Hn.T).max() < 1e-11
    # spin-flip symmetry of the synthetic block is absent, but left/right truncations of the mirrored superblock agree
    assert abs(btL.TruncErr - btR.TruncErr) < 1e-9


def test_error_codes(P, ctx):
    b = P.Block.Initialize(ctx, 2, [1.5, 0.5, -0.5, -1.5], [2, 3, 2, 1])
    with pytest.raises(P.DmrgxError) as e:
        b.set_operator(P.OpSz, 0, [0, 1, 1, 1, 1, 1, 1, 1, 1], [5], [1.0])  # row 0 (sector 0) -> column in sector 2
    assert e.value.code == 63
    with pytest.raises(P.DmrgxError):
        P.Block.Initialize(ctx, 2, [0.5, 0.5], [1, 1])
    with pytest.raises(P.DmrgxError) as e:
        b.set_operator(P.OpSz, 7, [0] * 9, [], [])
    assert e.value.code == 63


def test_exact_chain_sparse_workload_ground_state(P, ctx):
    """The sparse-sector path on the GPU (CSR / identity tiles, no tensor work): exact 8-site halves of the 16-site open
    Heisenberg chain; E0 from exact diagonalisation (SURVEY.md §8c)."""
    import bench_workload as W
    sw = W.ExactChainWorkload(P, ctx, 8)
    assert sw.n == 12870
    e, psi, st = sw.shell.EPSSolve(tol=1e-12)
    assert st["converged"] and abs(e - (-6.911737145575)) < 1e-9
    x = sw.random_state(4); y = sw.random_state(5)
    Hx = sw.shell.MatMult_host(x); Hy = sw.shell.MatMult_host(y)
    assert abs(y @ Hx - x @ Hy) < 1e-12


def test_correlator_operator_products_match_dense(P, ctx, orc):
    pc.check_correlator_products(P, orc, ctx, J1J2_CYL)


def test_testkron01_kronblocks_golden(P, ctx, golden_dir):
    pc.check_testkron01_kronblocks(P, ctx, golden_dir)


def test_testkron01_operator_rows_on_the_product(P, ctx, golden_dir):
    pc.check_testkron01_operator_rows(P, ctx, golden_dir)


def test_frozen_step_fixture(P, ctx, golden_dir):
    """the CUDA path against committed numbers (no oracle involved at test time)"""
    pc.check_step_fixture(P, ctx, golden_dir)


def test_wavefunction_prediction_extension(P, ctx):
    """csrc/predict.cpp on the device: exact overlap on un-truncated blocks (both growth directions), same energies and fewer
    H*psi on truncating sweeps"""
    pc.check_wavefunction_prediction(P, ctx)
