"""The three host-planned operations of a DMRG step, each against an extended-precision reference at its own edges:
eigs_smallest (EPSSolve: the thick-restart Lanczos), truncate (GetTruncation: ρ blocks, syevd, the top-m selection and the
gather of U) and rotate (RotateOperators: U_I·O[I,J]·U_Jᵀ and the Sm views).

The inputs are built from the Python API (Block.Initialize + set_operator, KronEye_Explicit) with a known answer: H with a
chosen spectrum in a hidden orthogonal basis, ψ with chosen Schmidt values per sector pair.  Products and residuals are formed
in long double; every bound is C·n·u·‖·‖ with the one constant C below, the same on both backends, and subspaces are compared
with a gap-aware (Davis–Kahan) bound.  The host code of all three operations also runs on the CPU emulation of the device
layer, so the plancheck flavour pins the host logic without a GPU."""
import numpy as np
import pytest

from devcheck_common import LD, U
from measure_common import P, ctx, SM, SZ, SP, kron_index  # noqa: F401  (fixtures)

C = 32                  # the constant of every c·n·u bound in this file
TOL = 1e-12             # -H_eps_tol of the solves
# csrc/dev.h GS_REFINE_REL: the second Gram-Schmidt correction is skipped when it is below 1e-12 of the vector, so a Lanczos
# vector may keep components of that relative size along the basis.  The true residual of a Ritz pair then differs from the
# solver's |β·s_last| by up to about GS_REFINE_REL·‖H‖ (seen: 1.2e-12 against 2.6e-17 at n = 40, ncv = 39), which is the
# accuracy floor of the solve next to c·n·u·‖H‖.
GS_REFINE_REL = 1e-12


# ---- building blocks --------------------------------------------------------------------------------------------------------

def csr(A):
    rp, col, val = [0], [], []
    for r in range(A.shape[0]):
        nz = np.nonzero(A[r])[0]
        col.extend(nz.tolist()); val.extend(A[r, nz].tolist()); rp.append(len(col))
    return rp, col, val


def block(P, ctx, qn, sizes, H=None, Sz=None, Sp=None, nsites=1):
    """a block with the given sectors and (one site's) operators; missing ones are zero"""
    b = P.Block.Initialize(ctx, nsites, qn, sizes)
    n = int(sum(sizes))
    Z = np.zeros((n, n))
    b.set_operator(P.OpH, 0, *csr(Z if H is None else H))
    b.set_operator(P.OpSz, 0, *csr(Z if Sz is None else Sz))
    b.set_operator(P.OpSp, 0, *csr(Z if Sp is None else Sp))
    return b


def hidden(rng, w):
    """Q·diag(w)·Qᵀ with a random orthogonal Q; returns (H, Q)"""
    Q, _ = np.linalg.qr(rng.standard_normal((len(w), len(w))))
    return (Q * w) @ Q.T, Q


def superblock_dense(P, kb, terms):
    """the superblock Hamiltonian of KronSumConstruct(terms) in long double, in the Kron's state order: H_L⊗1 + 1⊗H_R +
    Σ a·O_L⊗O_R from the blocks' own operators (right-block site n-1-s for superblock site s)"""
    L, R = kb.left, kb.right
    nL, n = L.NumSites(), L.NumSites() + R.NumSites()
    NL, NR = L.NumStates(), R.NumStates()

    def op(blk, o, i):
        return blk.get_operator_dense(P.OpSp, i).T if o == SM else blk.get_operator_dense(o, i)
    H = np.kron(L.get_operator_dense(P.OpH).astype(LD), np.eye(NR, dtype=LD)) + np.kron(np.eye(NL, dtype=LD), R.get_operator_dense(P.OpH).astype(LD))
    for a, io, i, jo, j in terms:
        assert i < nL <= j
        H += LD(a) * np.kron(op(L, io, i).astype(LD), op(R, jo, n - 1 - j).astype(LD))
    idx = kron_index(kb, NR)
    return H[np.ix_(idx, idx)]


def two_norm(A):
    return float(np.linalg.norm(np.asarray(A, dtype=float), 2))


# ---- 1. eigs_smallest ----------------------------------------------------------------------------------------------------------

def one_block_shell(P, ctx, H):
    """H as the left block's Hamiltonian, a one-state right block with H_R = 0 and no terms: the superblock matrix is H"""
    L = block(P, ctx, [0.0], [len(H)], H=H)
    R = block(P, ctx, [0.0], [1])
    kb = P.KronBlocks(L, R, [0.0])
    return kb, kb.KronSumConstruct([])


def check_solve(Hld, e, psi, st, tol=TOL, lam=None, what=""):
    """the checks every solve must pass; returns the long-double residual norm"""
    n = len(Hld)
    lam = np.linalg.eigvalsh(np.asarray(Hld, dtype=float)) if lam is None else lam
    normH = max(abs(lam[0]), abs(lam[-1]))
    slack = C * n * U * normH + 4 * GS_REFINE_REL * normH
    x = psi.get().astype(LD)
    assert abs(float(np.sqrt(x @ x)) - 1.0) <= C * n * U, (what, float(np.sqrt(x @ x)))
    r = Hld @ x - LD(e) * x
    rn = float(np.sqrt(r @ r))
    assert np.isfinite(e) and e >= lam[0] - slack, (what, e, lam[0])
    if st["converged"]:
        assert rn <= tol * abs(e) + slack, (what, rn, tol * abs(e), slack)
        # |β·s_last| is the residual norm of the Ritz pair in exact arithmetic
        assert abs(st["resid"] - rn) <= slack, (what, st["resid"], rn, slack)
        # an eigenvalue lies within ‖r‖ of θ: it must be λ₀ (and not λ₁ where the gap allows telling them apart)
        assert abs(e - lam[0]) <= rn + slack, (what, e, lam[0], rn)
        gap = lam[np.searchsorted(lam, lam[0] + slack, side="right")] - lam[0] if lam[-1] > lam[0] + slack else np.inf
        if gap > 2 * (rn + slack):
            assert abs(e - lam[0]) < gap / 2, (what, e, lam[:2])
    return rn


def bits(a):
    return np.asarray(a, dtype=np.float64).view(np.uint64)


SIZES = [(ng, ncv) for ncv in (1, 2, 16, 39) for ng in sorted({1, 2, 3, ncv - 1, ncv, ncv + 1, 2 * ncv + 1}) if ng >= 1]


@pytest.mark.parametrize("ng,ncv", SIZES)
def test_eigs_sizes(P, ctx, ng, ncv):
    """superblocks shorter than, as long as and longer than the basis, ncv = 1 (a basis of 2) up to the 39 of the fused kernels"""
    rng = np.random.default_rng([1, ng, ncv])
    w = np.sort(rng.uniform(-2.0, 1.0, ng))
    H, Q = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=ncv)
    assert st["converged"], st
    check_solve(H.astype(LD), e, psi, st, lam=w, what=(ng, ncv))
    if ng <= max(ncv, 2):   # the basis spans the whole space: one cycle, exact
        assert st["nrestart"] == 0 and st["nmatvec"] <= ng, st


def test_eigs_refuses_ncv_above_basis_limit(P, ctx):
    kb, sh = one_block_shell(P, ctx, np.diag(np.arange(50.0)))
    with pytest.raises(P.DmrgxError) as exc:
        sh.EPSSolve(tol=TOL, ncv=40)
    assert exc.value.code == 63


def spectrum(kind, rng):
    if kind == "separated":
        return np.sort(rng.uniform(-1.0, 1.0, 90)) + np.arange(90) * 0.05
    if kind == "degenerate2":
        w = np.sort(rng.uniform(-1.0, 1.0, 90)); w[:2] = -1.5
        return w
    if kind == "degenerate3":
        w = np.sort(rng.uniform(-1.0, 1.0, 90)); w[:3] = -1.5
        return w
    if kind == "gap1e-9":
        w = np.sort(rng.uniform(-1.0, 1.0, 33)); w[0] = -1.5; w[1] = -1.5 + 1e-9 * 1.5
        return w
    if kind == "clustered":
        return np.concatenate([-1.0 + 1e-3 * np.arange(6), np.sort(rng.uniform(-0.99, 1.0, 394))])
    if kind == "shifted":
        return np.sort(rng.uniform(-1.0, 1.0, 90)) - 1e4
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["separated", "degenerate2", "degenerate3", "gap1e-9", "clustered", "shifted"])
def test_eigs_spectra(P, ctx, kind):
    rng = np.random.default_rng([2, len(kind)])
    w = spectrum(kind, rng)
    H, Q = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=16)
    assert st["converged"], st
    rn = check_solve(H.astype(LD), e, psi, st, lam=w, what=kind)
    if kind.startswith("degenerate"):   # ψ lies in the eigenspace of λ₀
        d = int(kind[-1])
        x = psi.get()
        out = x - Q[:, :d] @ (Q[:, :d].T @ x)
        assert np.linalg.norm(out) <= (rn + C * len(w) * U * np.abs(w).max()) / (w[d] - w[0]), np.linalg.norm(out)
    if kind == "clustered":
        assert st["nrestart"] > 0, st


@pytest.mark.parametrize("scale", [1e-8, 1.0, 1e3, 1e6])
def test_eigs_breakdown_scales(P, ctx, scale):
    """three distinct eigenvalues, 40-fold each: the Krylov space of any start vector is three-dimensional.  The absolute
    1e-14 breakdown threshold is reached at ‖H‖ = 1e-8 and 1 (the solve then goes on from a fresh random direction) but not
    at 1e3 and 1e6, where it goes on along rounding noise: both paths must return the ground state."""
    rng = np.random.default_rng(3)
    w = np.repeat([-1.0, 0.25, 1.0], 40) * scale
    H, Q = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=16)
    assert st["converged"], st
    check_solve(H.astype(LD), e, psi, st, lam=w, what=scale)
    assert abs(e - w[0]) <= C * len(w) * U * abs(w[0]), (e, w[0])


def test_eigs_two_blocks_separable(P, ctx):
    """H_L⊗1 + 1⊗H_R: the spectrum is every sum λ_L + λ_R"""
    rng = np.random.default_rng(4)
    wl, wr = np.sort(rng.uniform(-1, 1, 23)), np.sort(rng.uniform(-1, 1, 17))
    HL, _ = hidden(rng, wl); HR, _ = hidden(rng, wr)
    kb = P.KronBlocks(block(P, ctx, [0.0], [23], H=HL), block(P, ctx, [0.0], [17], H=HR), [0.0])
    sh = kb.KronSumConstruct([])
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=16)
    lam = np.sort(np.add.outer(wl, wr).ravel())
    assert st["converged"]
    check_solve(superblock_dense(P, kb, []), e, psi, st, lam=lam)


def coupled_blocks(P, ctx, rng, nL=(9, 14), nR=(11, 7)):
    """two blocks with two sectors each (qn ±1/2), random symmetric H and Sz and a random Sp from sector -1/2 to +1/2"""
    def one(n):
        N = sum(n)
        H = rng.standard_normal((N, N)); H = H + H.T
        Sz = np.zeros((N, N)); Sp = np.zeros((N, N))
        a, b = n         # sector +1/2 (a states) first: the sectors go in descending order
        S = rng.standard_normal((a, a)); Sz[:a, :a] = S + S.T
        S = rng.standard_normal((b, b)); Sz[a:, a:] = S + S.T
        H[:a, a:] = 0; H[a:, :a] = 0
        Sp[:a, a:] = rng.standard_normal((a, b))
        return block(P, ctx, [0.5, -0.5], list(n), H=H, Sz=Sz, Sp=Sp)
    return one(nL), one(nR)


@pytest.mark.parametrize("fill", [0.0, 2.0])
def test_eigs_coupled_blocks(P, ctx, fill):
    """Sz·Sz and S+S- + S-S+ couplings between the blocks (H not separable), dense (fill 0) and CSR (fill 2) tiles"""
    ctx.set_dense_threshold(fill)
    rng = np.random.default_rng(5)
    L, R = coupled_blocks(P, ctx, rng)
    kb = P.KronBlocks(L, R, [0.0])
    terms = [(0.7, SZ, 0, SZ, 1), (0.35, SP, 0, SM, 1), (0.35, SM, 0, SP, 1)]
    sh = kb.KronSumConstruct(terms)
    Hld = superblock_dense(P, kb, terms)
    x = rng.standard_normal(sh.n)
    y = sh.MatMult_host(x)
    assert np.abs(y - np.asarray(Hld @ x.astype(LD), dtype=float)).max() <= C * sh.n * U * two_norm(Hld) * np.abs(x).max()
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=16)
    assert st["converged"]
    check_solve(Hld, e, psi, st)


def test_eigs_max_it_runs_out(P, ctx):
    """one restart cycle on a slowly converging spectrum: not converged, θ is still a Ritz value (the Rayleigh quotient of ψ)
    and not below λ₀"""
    rng = np.random.default_rng(6)
    w = spectrum("clustered", rng)
    H, _ = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=8, max_it=1)
    assert not st["converged"] and st["nmatvec"] == 8, st
    check_solve(H.astype(LD), e, psi, st, lam=w)
    x = psi.get().astype(LD)
    assert abs(float(x @ (H.astype(LD) @ x)) - e) <= C * len(w) * U * np.abs(w).max()


def test_eigs_in_cycle_stopping_test(P, ctx, monkeypatch):
    """the stopping test inside the cycle (on above DMRGX_EARLY_TEST_MIN) gives the same eigenpair to tol as the test at the
    restart boundary only"""
    rng = np.random.default_rng(7)
    w = spectrum("separated", rng)
    H, _ = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    out = {}
    for on in (True, False):
        monkeypatch.setenv("DMRGX_EARLY_TEST_MIN", "1" if on else str(10 ** 12))
        e, psi, st = sh.EPSSolve(tol=TOL, ncv=16)
        assert st["converged"]
        check_solve(H.astype(LD), e, psi, st, lam=w, what=on)
        out[on] = (e, psi.get(), st)
    (ea, xa, sa), (eb, xb, sb) = out[True], out[False]
    assert abs(ea - eb) <= 2 * TOL * abs(eb)
    assert 1.0 - abs(xa @ xb) <= 2 * TOL * abs(eb) / (w[1] - w[0])
    assert sa["nmatvec"] <= sb["nmatvec"]


def test_eigs_unusable_start_vectors_take_the_random_one(P, ctx):
    """a zero, NaN or Inf start vector gives the seeded random solve bit for bit; and two solves give the same bits"""
    rng = np.random.default_rng(8)
    w = spectrum("separated", rng)
    H, _ = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    e0, p0, s0 = sh.EPSSolve(tol=TOL, ncv=16, seed=99)
    e1, p1, s1 = sh.EPSSolve(tol=TOL, ncv=16, seed=99)
    assert bits(e0) == bits(e1) and np.array_equal(bits(p0.get()), bits(p1.get())) and s0 == s1
    for bad in (np.zeros(len(w)), np.full(len(w), np.nan), np.where(np.arange(len(w)) == 3, np.inf, 1.0)):
        e, p, s = sh.EPSSolve(tol=TOL, ncv=16, seed=99, initial=ctx.vec(len(w), bad))
        assert bits(e) == bits(e0) and np.array_equal(bits(p.get()), bits(p0.get())) and s == s0


def test_eigs_start_exact_ground_state(P, ctx):
    rng = np.random.default_rng(9)
    w = spectrum("separated", rng)
    H, Q = hidden(rng, w)
    kb, sh = one_block_shell(P, ctx, H)
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=16, initial=ctx.vec(len(w), Q[:, 0]))
    assert st["converged"] and st["nrestart"] == 0, st
    check_solve(H.astype(LD), e, psi, st, lam=w)


@pytest.mark.parametrize("start,ncv", [("excited", 8), ("excited", 16), ("excited", 39), ("invariant", 16), ("invariant", 39)])
def test_eigs_start_without_ground_state(P, ctx, start, ncv):
    """dmrgx_eigs_smallest_from returns the ground state also from a start vector with no component along it: an exact excited
    eigenvector of H, or a vector of an exactly invariant subspace, the 7 states of a block of H (eigenvalues 3..9) that
    a hidden permutation scatters over the basis, as a symmetry sector would.  Its Krylov space breaks down before the basis
    is full, and the solve must go on instead of reporting the lowest Ritz pair of that space.
    (The new direction gets the rest of the cycle, ncv minus the dimension of the exhausted space steps; with one or two
    steps left it cannot find a Ritz value below that pair, which is why the 7-dimensional case runs at ncv >= 16.  The block
    structure is exact in floating point: in a dense orthogonal basis the subspace is invariant only to rounding, Lanczos
    amplifies the rounding-sized ground-state component, and the outcome depends on that noise.)"""
    rng = np.random.default_rng([10, ncv])
    w = np.linspace(-1.0, 1.0, 60)
    if start == "excited":
        H, Q = hidden(rng, w)
        g = Q[:, 5]
    else:
        inv, rest = np.arange(3, 10), np.setdiff1d(np.arange(60), np.arange(3, 10))
        perm = rng.permutation(60)
        H = np.zeros((60, 60))
        H[np.ix_(perm[:7], perm[:7])] = hidden(rng, w[inv])[0]
        H[np.ix_(perm[7:], perm[7:])] = hidden(rng, w[rest])[0]
        g = np.zeros(60)
        g[perm[:7]] = rng.standard_normal(7)
    kb, sh = one_block_shell(P, ctx, H)
    e, psi, st = sh.EPSSolve(tol=TOL, ncv=ncv, initial=ctx.vec(len(w), g))
    assert st["converged"], st
    check_solve(H.astype(LD), e, psi, st, lam=w, what=start)
    assert abs(e - w[0]) <= 1e-10, (e, w[0])


# ---- 2. GetTruncation ----------------------------------------------------------------------------------------------------------

def orth(rng, n, k):
    """n×k with orthonormal columns"""
    if k == 0:
        return np.zeros((n, 0))
    Q, _ = np.linalg.qr(rng.standard_normal((n, k)))
    return Q


class Schmidt:
    """ψ of a Kron with X_p = U_p·diag(s_p)·V_pᵀ on every sector pair; s chosen in long double, normalised over all pairs"""

    def __init__(self, kb, rng, svals):
        """svals(p, nL, nR): the Schmidt values of sector pair p (Kron order) of nL × nR"""
        qn, il, ir, sz, off = kb.data()
        self.kb, self.il, self.ir, self.off = kb, il, ir, off
        Lq, Ls = kb.left.sectors(); Rq, Rs = kb.right.sectors()
        svals = [svals(p, int(Ls[il[p]]), int(Rs[ir[p]])) for p in range(len(qn))]
        norm = np.sqrt(sum((np.asarray(s, dtype=LD) ** 2).sum() for s in svals))
        self.s = [np.asarray(s, dtype=LD) / norm for s in svals]
        self.U, self.V, self.X = [], [], []
        psi = np.zeros(int(off[-1]))
        for p in range(len(qn)):
            nL, nR = int(Ls[il[p]]), int(Rs[ir[p]])
            k = len(self.s[p]); assert k <= min(nL, nR)
            Up, Vp = orth(rng, nL, k), orth(rng, nR, k)
            X = (Up * np.asarray(self.s[p], dtype=float)) @ Vp.T
            psi[off[p]:off[p + 1]] = X.ravel()
            self.U.append(Up); self.V.append(Vp); self.X.append(X)
        self.psi = psi
        self.dims = {True: [int(Ls[i]) for i in il], False: [int(Rs[i]) for i in ir]}

    def spectrum(self, left):
        """per pair, descending: s² and zeros up to the block dimension"""
        out = []
        for p, s in enumerate(self.s):
            n = self.dims[left][p]
            out.append(np.concatenate([np.sort(s ** 2)[::-1], np.zeros(n - len(s), dtype=LD)]))
        return out


def select(spec, blk, m):
    """the reference's rule: (eigval, seq, blk) per pair in descending order, stable sort by -eigval, the first m, stable sort
    by block; returns {block: kept count} and the kept eigenvalues"""
    ent = [(float(v), p, blk[p]) for p, sp in enumerate(spec) for v in sp]
    ent = sorted(ent, key=lambda t: -t[0])[:m]
    ent = sorted(ent, key=lambda t: t[2])
    kept = {}
    for _, _, b in ent:
        kept[b] = kept.get(b, 0) + 1
    return kept, [v for v, _, _ in ent]


def check_side(P, bt, sch, left, m, skip_projector_blocks=(), what=""):
    kb = sch.kb
    blkidx = sch.il if left else sch.ir
    blk_sizes = (kb.left if left else kb.right).sectors()[1]
    ref = sch.spectrum(left)
    nmax = max(max(sch.dims[True]), max(sch.dims[False]), 1)
    # spectrum(): per pair, descending, with the pair's block index
    ev, bi = bt.spectrum()
    assert bi.tolist() == [int(blkidx[p]) for p in range(len(ref)) for _ in ref[p]], what
    pos = 0
    for p, r in enumerate(ref):
        got = ev[pos:pos + len(r)]; pos += len(r)
        bound = C * nmax * U * float(r.max() if len(r) else 0.0) + C * nmax * U * float(max(x.max() for x in ref)) * (float(r.max()) == 0.0)
        assert np.abs(got.astype(LD) - r).max() <= max(bound, C * nmax * U * 1e-300), (what, p, float(np.abs(got - r).max()), bound)
    # kept counts per sector: exactly the reference's where the cut has a gap; inside a tie that rounding can reorder (the
    # zero-weight states past the rank) only the states above the tie are fixed
    kept, kept_vals = select(ref, [int(b) for b in blkidx], m)
    q, sz = bt.sectors()
    allq = list((kb.left if left else kb.right).sectors()[0])
    got = {allq.index(qq): int(n) for qq, n in zip(q.tolist(), sz.tolist())}
    flat = np.sort(np.concatenate(ref).astype(float))[::-1]
    eps = 2 * C * nmax * U * float(flat[0])
    if m >= len(flat) or flat[m - 1] - flat[m] > eps:
        assert got == kept, (what, got, kept)
    else:
        tie = flat[m - 1]
        for b in set(int(x) for x in blkidx):
            above = sum(int((r > tie + eps).sum()) for p, r in enumerate(ref) if blkidx[p] == b)
            assert got.get(b, 0) >= above, (what, b, got, kept)
        assert sum(got.values()) == min(m, len(flat)), (what, got)
        kept = got
        kept_vals = [v for b in got for v in sorted([float(x) for p, r in enumerate(ref) if blkidx[p] == b for x in r], reverse=True)[:got[b]]]
    assert bt.m == sum(kept.values())
    # TruncErr bit for bit from the returned spectrum under the same rule (the kept positive eigenvalues, subtracted from 1 in
    # block order): only the rounding-sized negative eigenvalues of a rank-deficient ρ tell "positive" apart
    sel = sorted(((float(v), int(b)) for v, b in zip(ev, bi)), key=lambda t: -t[0])[:m]
    te = 1.0
    for v, _ in sorted(sel, key=lambda t: t[1]):
        te -= (v > 0) * v
    assert bits(bt.TruncErr) == bits(te), (what, bt.TruncErr, te)
    # TruncErr = 1 - Σ of the kept positive eigenvalues
    te = 1.0 - sum(LD(v) for v in kept_vals if v > 0)
    assert abs(bt.TruncErr - float(te)) <= C * nmax * U, (what, bt.TruncErr, float(te))
    # U: orthonormal rows, each block's rows inside its sector's columns, the right projector where the cut has a gap
    Ut = bt.RotMatT()
    assert np.abs(Ut @ Ut.T - np.eye(bt.m)).max() <= C * nmax * U, what
    offs = np.concatenate([[0], np.cumsum(blk_sizes)])
    row = 0
    for b in sorted(kept):
        k = kept[b]
        Ub = Ut[row:row + k]; row += k
        assert not np.any(np.delete(Ub, np.s_[offs[b]:offs[b + 1]], axis=1)), (what, b)
        if b in skip_projector_blocks:
            continue
        p = [pp for pp in range(len(ref)) if blkidx[pp] == b][0]
        s2 = ref[p]
        W = sch.U[p] if left else sch.V[p]
        r = len(sch.s[p])
        kk = min(k, r)
        Pb = Ub[:, offs[b]:offs[b + 1]].T @ Ub[:, offs[b]:offs[b + 1]]
        if kk == k:     # the kept span is spanned by the leading Schmidt vectors (ties at the cut excluded by the caller)
            gap = float(s2[k - 1] - (s2[k] if k < len(s2) else 0.0))
            if gap > 0:
                Pref = W[:, :k] @ W[:, :k].T
                assert two_norm(Pb - Pref) <= C * nmax * U * float(s2[0]) / gap, (what, b, two_norm(Pb - Pref), gap)
        elif r > 0:     # zero-weight states kept: the span holds every nonzero Schmidt vector
            Wr = W[:, :r]
            assert np.linalg.norm(Wr - Pb @ Wr, 2) <= C * nmax * U * float(s2[0]) / float(s2[r - 1]), (what, b)


def two_sided_blocks(P, ctx, pairs):
    """blocks whose sectors pair up one to one under qn 0: L sector k (qn k) of pairs[k][0] states with R sector -k of
    pairs[k][1] states"""
    qn = [float(k) for k in range(len(pairs))][::-1]
    L = P.Block.Initialize(ctx, 1, qn, [a for a, _ in pairs][::-1])
    R = P.Block.Initialize(ctx, 1, [-q for q in qn][::-1], [b for _, b in pairs])
    return P.KronBlocks(L, R, [0.0])


def graded(rng, k, lo=1e-3):
    """k distinct Schmidt values between 1 and lo, well separated relative to the bounds"""
    return np.sort(np.exp(np.linspace(0.0, np.log(lo), k)) * (1 + 0.01 * rng.uniform(size=k)))[::-1]


TRUNC_SHAPES = {   # (nL, nR) of each sector pair; ρ_L has size nL and K = nR, ρ_R size nR and K = nL
    "edges": [(1, 1), (63, 64), (64, 63), (65, 2), (3, 65), (193, 7)],
    "long_K": [(64, 193), (65, 1), (1, 64)],
    "cuda_large": [(833, 2048), (193, 833)],
}


@pytest.mark.parametrize("shape", list(TRUNC_SHAPES))
def test_truncation_block_sizes(P, ctx, shape):
    """ρ blocks on both sides of the 64-state switch of the eigensolver, 193 and 833, with contraction lengths from 1 to
    several thousand; rank-deficient ρ on the longer side of every pair"""
    if shape == "cuda_large" and P.kind != "cuda":
        pytest.skip("the 833-state blocks are checked on the CUDA build (minutes on the emulation)")
    rng = np.random.default_rng(len(shape))
    pairs = TRUNC_SHAPES[shape]
    kb = two_sided_blocks(P, ctx, pairs)
    sch = Schmidt(kb, rng, lambda p, nL, nR: graded(rng, min(nL, nR)) * (0.5 + p))
    rank = sum(len(s) for s in sch.s)
    for m in (1, rank // 2, rank, rank + 1):
        btL, btR = P.GetTruncation(kb, ctx.vec(len(sch.psi), sch.psi), m)
        check_side(P, btL, sch, True, m, what=(shape, m, "L"))
        check_side(P, btR, sch, False, m, what=(shape, m, "R"))


def test_truncation_m_edges_and_zero_pairs(P, ctx):
    """pairs where ψ is identically zero, m = 1, m at and above the rank, m above every state, and m = 0"""
    rng = np.random.default_rng(11)
    pairs = [(5, 9), (7, 7), (4, 6), (6, 3)]
    kb = two_sided_blocks(P, ctx, pairs)
    sch = Schmidt(kb, rng, lambda p, nL, nR: [graded(rng, 3), [], graded(rng, 3) * 0.3, []][p])
    d = ctx.vec(len(sch.psi), sch.psi)
    total = sum(a for a, _ in pairs)
    for m in (1, 3, 7, 8, total, total + 10):
        btL, btR = P.GetTruncation(kb, d, m)
        # the zero-weight states kept past the rank are an arbitrary basis of a null space: no projector there
        check_side(P, btL, sch, True, m, what=("L", m))
        check_side(P, btR, sch, False, m, what=("R", m))
    with pytest.raises(P.DmrgxError):
        P.GetTruncation(kb, d, 0)


def test_truncation_cut_inside_multiplet(P, ctx):
    """the cut falls inside a 4-fold multiplet of one block: the count follows the reference's stable order, and the kept span
    is checked only where there is a gap"""
    rng = np.random.default_rng(12)
    pairs = [(9, 9), (8, 10)]
    kb = two_sided_blocks(P, ctx, pairs)
    s0 = np.array([1.0, 0.8, 0.6, 0.6, 0.6, 0.6, 0.1])
    sch = Schmidt(kb, rng, lambda p, nL, nR: [s0, np.array([0.9, 0.5, 0.05])][p])
    btL, btR = P.GetTruncation(kb, ctx.vec(len(sch.psi), sch.psi), 6)
    for bt, left in ((btL, True), (btR, False)):
        q, sz = bt.sectors()
        assert sz.sum() == 6 and bt.m == 6
        # 1.0, 0.9, 0.8 and then three of the four 0.6: all from block 0, whose multiplet is cut
        b0 = int((sch.il if left else sch.ir)[0])
        check_side(P, bt, sch, left, 6, skip_projector_blocks=(b0,), what=left)
        assert sz[q.tolist().index(allq(kb, left)[b0])] == 5
        # the kept span of the cut block: it holds the two leading Schmidt vectors and lies inside the span of the first six
        Ub = block_rows(bt, kb, left, b0)
        W = sch.U[0] if left else sch.V[0]
        s2 = np.asarray(sch.s[0], dtype=float) ** 2
        Pb = Ub.T @ Ub
        bound = C * 20 * U * s2[0]
        assert np.linalg.norm(W[:, :2] - Pb @ W[:, :2], 2) <= bound / (s2[1] - s2[2])
        assert np.linalg.norm(Ub.T - W[:, :6] @ (W[:, :6].T @ Ub.T), 2) <= bound / (s2[5] - s2[6])


def allq(kb, left):
    return list((kb.left if left else kb.right).sectors()[0])


def block_rows(bt, kb, left, b):
    """the rows of RotMatT that belong to block sector b, restricted to that sector's columns"""
    q, sz = bt.sectors()
    k = q.tolist().index(allq(kb, left)[b])
    r0 = int(sz[:k].sum())
    offs = np.concatenate([[0], np.cumsum((kb.left if left else kb.right).sectors()[1])])
    return bt.RotMatT()[r0:r0 + int(sz[k]), offs[b]:offs[b + 1]]


def test_truncation_cross_block_tie_is_stable(P, ctx):
    """six pairs with identical X (40 × 40, 240 states in 40 six-fold ties): their ρ spectra are bit-identical, so a cut inside
    a cross-block tie keeps the states of the pairs that come first, as the reference's stable sort does.  (With fewer than
    17 states an unstable std::sort still sorts by insertion and would keep the same ones.)"""
    rng = np.random.default_rng(13)
    ncopy, n = 6, 40
    kb = two_sided_blocks(P, ctx, [(n, n)] * ncopy + [(6, 6)])
    s = graded(rng, n, 0.3)
    sch = Schmidt(kb, rng, lambda p, nL, nR: s if nL == n else 0.01 * graded(rng, 3))
    qn, il, ir, sz, off = kb.data()
    copies = [p for p in range(len(qn)) if sz[p] == n * n]
    psi = sch.psi.copy()
    for p in copies[1:]:
        psi[off[p]:off[p + 1]] = psi[off[copies[0]]:off[copies[0] + 1]]
    m = ncopy * 7 + 3     # the seven largest values of every copy, then three of the six-fold tie at the eighth
    btL, btR = P.GetTruncation(kb, ctx.vec(len(psi), psi), m)
    for bt, left in ((btL, True), (btR, False)):
        ev, bi = bt.spectrum()
        start = [int(np.sum(np.where(np.arange(len(qn)) < p, [int(x) for x in sch.dims[left]], 0))) for p in copies]
        for a in start[1:]:
            assert np.array_equal(bits(ev[a:a + n]), bits(ev[start[0]:start[0] + n])), left
        blk = [int(b) for b in (sch.il if left else sch.ir)]
        want = {blk[p]: 7 + (k < 3) for k, p in enumerate(copies)}
        q, sz_ = bt.sectors()
        assert {allq(kb, left).index(qq): int(c) for qq, c in zip(q.tolist(), sz_.tolist())} == want, (left, q, sz_)


def test_truncation_refuses_sector_in_two_pairs(P, ctx):
    """a block sector that appears in two sector pairs of the target: not supported, code 56"""
    L = P.Block.Initialize(ctx, 1, [1.0, 0.0], [3, 3])
    R = P.Block.Initialize(ctx, 1, [1.0, 0.0, -1.0], [3, 3, 3])
    kb = P.KronBlocks(L, R, [0.0, 1.0])
    n = kb.NumStates()
    x = np.random.default_rng(14).standard_normal(n); x /= np.linalg.norm(x)
    with pytest.raises(P.DmrgxError) as exc:
        P.GetTruncation(kb, ctx.vec(n, x), n)
    assert exc.value.code == 56


# ---- 3. RotateOperators --------------------------------------------------------------------------------------------------------

CHAIN = dict(Lx=12, Ly=1, J1=0.5, Jz1=1.0, J2=0.0, Jz2=0.0, bcx=0, bcy=0)


def chain_terms(P, k):
    h = CHAIN
    return P.HamiltonianTerms(h["Lx"], h["Ly"], h["J1"], h["Jz1"], h["J2"], h["Jz2"], k, h["bcx"], h["bcy"])


def enlarged(P, ctx, nsites):
    """the exact (nsites - 1)-site chain block enlarged by one site: EYE tiles from KronEye_Explicit, and dense or CSR tiles
    for the rest by the context's threshold"""
    site = P.Block.SingleSite(ctx)
    blk = P.Block.SingleSite(ctx)
    for k in range(2, nsites):
        blk = P.KronEye_Explicit(blk, site, chain_terms(P, k))
    return P.KronEye_Explicit(blk, site, chain_terms(P, nsites))


def rotation_case(P, ctx, rng):
    """5 + 5 sites, target Sz = 0: the left sectors -5/2 .. 5/2 (sizes 1 5 10 10 5 1).  ψ is zero on the pair of left sector
    -1/2 (dropped: a gap in the middle of the new sector list) and rank one on the pairs of ±3/2 (one kept state each)"""
    L = enlarged(P, ctx, 5)
    kb = P.KronBlocks(L, L, [0.0])
    qn, il, ir, sz, off = kb.data()
    Lq, Ls = L.sectors()
    def svals(p, nL, nR):
        q = Lq[il[p]]
        return [] if q == -0.5 else graded(rng, 1) if abs(q) == 1.5 else graded(rng, min(nL, nR), 1e-2) * (1 + q)
    sch = Schmidt(kb, rng, svals)
    m = sum(len(s) for s in sch.s)
    btL, btR = P.GetTruncation(kb, ctx.vec(len(sch.psi), sch.psi), m)
    q, s = btL.sectors()
    assert -0.5 not in q.tolist() and 0.5 in q.tolist() and s[q.tolist().index(1.5)] == 1, (q, s)
    return L, kb, btL, btR


@pytest.mark.parametrize("fill", [0.0, 2.0])
def test_rotation_against_reference(P, ctx, fill):
    """every Sz_i, Sp_i and H of the rotated block against U·O·Uᵀ in long double; Sm = Spᵀ exactly; CheckOperatorBlocks"""
    ctx.set_dense_threshold(fill)
    rng = np.random.default_rng(15)
    L, kb, btL, btR = rotation_case(P, ctx, rng)
    Ut = btL.RotMatT()
    new = P.RotateOperators(L, btL)
    assert new.CheckOperatorBlocks() == 0
    assert new.NumStates() == btL.m and new.NumSites() == L.NumSites()
    q, s = new.sectors(); bq, bs = btL.sectors()
    assert q.tolist() == bq.tolist() and s.tolist() == bs.tolist()
    n = L.NumStates()
    for op, i in [(P.OpH, 0)] + [(o, i) for i in range(L.NumSites()) for o in (P.OpSz, P.OpSp)]:
        O = L.get_operator_dense(op, i)
        ref = Ut.astype(LD) @ O.astype(LD) @ Ut.T.astype(LD)
        got = new.get_operator_dense(op, i)
        bound = C * n * U * two_norm(O)
        assert np.abs(got.astype(LD) - ref).max() <= bound, (op, i, float(np.abs(got - ref).max()), bound)
        if op == P.OpSp:
            assert np.array_equal(new.get_operator_dense(P.OpSm, i), got.T), i


@pytest.mark.parametrize("fill", [0.0, 2.0])
def test_rotated_superblock_matvec(P, ctx, fill):
    """a superblock of two rotated blocks (each with a dropped middle sector): its H·ψ matches the long-double dense H built
    from the rotated operators, which pins the sector index shifts across the gap"""
    ctx.set_dense_threshold(fill)
    rng = np.random.default_rng(16)
    L, kb, btL, btR = rotation_case(P, ctx, rng)
    A = P.RotateOperators(L, btL)
    B = P.RotateOperators(L, btR)
    site = P.Block.SingleSite(ctx)
    A2 = P.KronEye_Explicit(A, site, chain_terms(P, 6))
    kb2 = P.KronBlocks(A2, B, [1.5, 0.5, -0.5])
    terms = [t for t in chain_terms(P, 11) if (t[2] < 6) != (t[4] < 6)]
    sh = kb2.KronSumConstruct(terms)
    Hld = superblock_dense(P, kb2, terms)
    for _ in range(2):
        x = rng.standard_normal(sh.n)
        y = sh.MatMult_host(x)
        bound = C * sh.n * U * two_norm(Hld) * np.abs(x).max()
        assert np.abs(y.astype(LD) - Hld @ x.astype(LD)).max() <= bound
