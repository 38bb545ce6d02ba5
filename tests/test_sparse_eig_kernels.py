"""Kernel-level tests of the two device-layer entry points test_device_kernels.py leaves out: run_spmm (spmm_kernel, the
sparse-sector H·ψ of exact blocks) and syevd_batch (cyclic Jacobi up to 64 states, batched block Jacobi above), each
called directly through the test-only shim tests/devcheck/devcheck.cpp (dc_spmm, dc_syevd) on two backends: `host` (the
host emulation tests/plancheck/dev_host.cpp) and `cuda` (the product's own sm_100a object; marked gpu).  Guard bands,
NaN operand padding, sentinel outputs and the longdouble reference follow test_device_kernels.py.

run_spmm.  Plans are built here, seeded, at the shapes where spmm_kernel branches: the TMA stage's head and tail patches
(tile offsets even and odd, nrows·nR odd and even, nrows·nR = 1 and 2), partial tiles (nrows < SP_ROWS: rows past them
are read by the kernel and must stay unwritten), the a-slot / s-slot batch of 24 and the b-slot batch of 8, the column
super-chunk loop of 1024 (nR up to 3072), all_in gathers next to L2 gathers in one tile, ELL padding mixed in, W = 0 and
ld > nR.  Source rows in L2 are scattered through X with NaN between them; every tile's staged range has NaN right
before and after it; Y is sentinel everywhere and keeps it outside the rows the tiles own.  An output element is a sum of

    N = na + ns + Σ_b 2·W_b

rounded products (an a- or s-term w·x is one product, a b-term (w·val)·x is two), checked against the longdouble sum
with |got - ref| <= (N + 2)·2^-53·Σ|terms|.  spmm_kernel sums every element in a fixed order that depends only on its
own tile, so two calls, the same tiles in reversed or shuffled list order (the planner reorders tiles), and a tile alone
or inside a batch of 640 all give the same bits.

syevd_batch.  Blocks sit at chosen element offsets of one pool, on bases 8 and 0 mod 16, in an order unrelated to their
size, with guards of 4 KiB between them; inputs are uploaded asynchronously on the main stream right before the call.
With u = 2^-53, ‖A‖ the spectral norm and c = 32, every block must satisfy

    eigenvalues    |w_k - eigvalsh(A)_k|     <= min(c·n·u, 5e-14)·‖A‖
    orthogonality  max |V Vᵀ - I|              <= min(c·n·u, 1e-12)
    residuals      ‖A v_k - w_k v_k‖₂          <= c·n·u·‖A‖
    graded ρ       ‖V_mᵀV_m - Q_m Q_mᵀ‖₂        <= c·n·u·‖A‖/gap     (V_m: the rows of the m largest eigenvalues)

with residuals, orthogonality and the projector computed in longdouble.  The caps are the fixed tolerances of
test_gpu_parity.py's eigensolver test, so neither bound is looser than those at any size; below n = 14 and 281 the c·n·u
term is the tighter one.  That test bounds max |V A Vᵀ - diag(w)| by 2e-13·‖A‖, which it still does; the residual norm
here is not capped, because the block path stops rotating a 64×64 sub-problem once its off-diagonal weight is below
3e-14·‖A‖_F, and for an indefinite spectrum ‖A‖_F grows like √n·‖A‖ (n = 832 on a B200: 2.9e-13·‖A‖).  Measured on a
B200 at a 1000 W power limit, the largest ratios to n·u are about 11 for the cyclic Jacobi's orthogonality and 10 for the block path's residuals.

Diagonal inputs, ties included, are exact on both paths (no rotation, only products with 1 and 0): w = sort(diag) and
row k is the unit vector of the k-th index of a stable argsort, bit for bit.  Guards must keep their bits and two calls
give the same bits.

Sizes: 1, 2, 63, 64, 65, 127, 128, 129, 192 and 193 on both backends (both sides of the 64 switch and of the 64-padding
of the block path); the cuda backend also runs 257, 512 and 832.
"""
import numpy as np
import pytest

from devcheck_common import (LD, SENT, SP_ASLOT, SP_BSLOT, SP_MAX_NR, SP_ROWS, SP_SSLOT, SP_TILE, U, Backend, assert_bound, bits, guard_for,
                             lib_path, rho_like, rng_for, with_spectrum)


@pytest.fixture(scope="module", params=["host", pytest.param("cuda", marks=pytest.mark.gpu)])
def dc(request):
    return Backend(request.param, lib_path(request.param))


# ---------------------------------------------------------------------------------------------------------------------
#  run_spmm
# ---------------------------------------------------------------------------------------------------------------------
NRS = [1, 2, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 2048, 2049, 3071, 3072]
SLOT_COUNTS = [0, 1, 23, 24, 25, 48, 49]       # a- and s-slots: around the batch of SP_AMAX = 24
BSLOT_COUNTS = [0, 1, 7, 8, 9, 16, 17]         # b-slots: around the batch of SP_BMAX = 8
WS = [0, 1, 5]


def _ceil32(n):
    return (n + 31) // 32 * 32


class SpPlan:
    """X (NaN between everything), the ELL pools I / V and the slot lists of a batch of tiles"""

    def __init__(self, rng):
        self.rng = rng
        self.x, self.nx = [], 0
        self.ints, self.ni = [], 0
        self.vals, self.nv = [], 0
        self.tiles, self.aslots, self.sslots, self.bslots = [], [], [], []

    def _put(self, arr, parity=None):
        """store arr in X after 1-3 NaN, at an offset of the given parity (random when None)"""
        gap = int(self.rng.integers(1, 4))
        if parity is None:
            parity = int(self.rng.integers(2))
        if (self.nx + gap) % 2 != parity:
            gap += 1
        self.x.append(np.full(gap, np.nan)); self.nx += gap
        off = self.nx
        self.x.append(np.asarray(arr, np.float64)); self.nx += len(arr)
        return off

    def _put_ell(self, cols, vals):
        pad = int(self.rng.integers(1, 3))
        self.ints.append(np.zeros(pad, np.int32)); self.vals.append(np.full(pad, np.nan))
        self.ni += pad; self.nv += pad
        oi, ov = self.ni, self.nv
        self.ints.append(cols.astype(np.int32).ravel()); self.vals.append(vals.ravel())
        self.ni += cols.size; self.nv += vals.size
        return oi, ov

    def _weights(self):
        w = self.rng.standard_normal(SP_ROWS)
        w[self.rng.random(SP_ROWS) < 0.15] = 0.0        # rows with fewer entries carry w = 0
        return w

    def _ell(self, nR, W, ld, ncols):
        """W slots of ld entries; columns past nR hold NaN values (never read); a quarter of the entries are padding"""
        cols = np.zeros((W, ld), np.int64)
        vals = np.full((W, ld), np.nan)
        if W:
            cols[:, :nR] = self.rng.integers(0, ncols, (W, nR))
            vals[:, :nR] = self.rng.standard_normal((W, nR))
            padm = self.rng.random((W, nR)) < 0.25
            cols[:, :nR][padm] = 0
            vals[:, :nR][padm] = 0.0
        return cols, vals

    def tile(self, nR, nrows, parity, na, ns, nb, ld_mode=0, all_in_first=0):
        rng = self.rng
        off = self._put(rng.standard_normal(nrows * nR), parity)
        self.x.append(np.full((SP_ROWS - nrows) * nR, np.nan)); self.nx += (SP_ROWS - nrows) * nR   # rows past a partial tile
        srcs = [self._put(rng.standard_normal(nR)) for _ in range(min(na, 6) + 1)]
        nRq = max(1, nR // 2 + 3)
        bsrcs = [self._put(rng.standard_normal(nRq)) for _ in range(3)]
        t = np.zeros(1, SP_TILE)[0]
        t["off"], t["nR"], t["nrows"] = off, nR, nrows
        t["a_begin"], t["a_count"] = len(self.aslots), na
        for _ in range(na):
            s = np.zeros(1, SP_ASLOT)[0]
            s["src"] = [srcs[int(rng.integers(len(srcs)))] for _ in range(SP_ROWS)]
            s["w"] = self._weights()
            self.aslots.append(s)
        t["s_begin"], t["s_count"] = len(self.sslots), ns
        for _ in range(ns):
            s = np.zeros(1, SP_SSLOT)[0]
            s["roff"] = rng.integers(0, nrows, SP_ROWS) * nR
            s["w"] = self._weights()
            self.sslots.append(s)
        t["b_begin"], t["b_count"] = len(self.bslots), nb
        for k in range(nb):
            s = np.zeros(1, SP_BSLOT)[0]
            W = WS[(k + ld_mode) % 3]
            ld = [nR, _ceil32(nR), _ceil32(nR) + 32, nR + 37][(k + ld_mode) % 4]
            s["all_in"] = (k + all_in_first) % 2
            if s["all_in"]:
                s["roff"] = rng.integers(0, nrows, SP_ROWS) * nR
                cols, vals = self._ell(nR, W, ld, nR)
            else:
                s["src"] = [bsrcs[int(rng.integers(len(bsrcs)))] for _ in range(SP_ROWS)]
                cols, vals = self._ell(nR, W, ld, nRq)
            s["W"], s["ld"] = W, ld
            s["ecol"], s["eval"] = self._put_ell(cols, vals)
            s["w"] = self._weights()
            self.bslots.append(s)
        self.tiles.append(t)

    def finish(self, g):
        self._put(np.zeros(0))
        self.X = np.concatenate([np.full(g, np.nan)] + self.x + [np.full(g, np.nan)])
        self.I = np.concatenate([np.zeros(g, np.int32)] + self.ints + [np.zeros(g + 1, np.int32)])
        self.V = np.concatenate([np.full(g, np.nan)] + self.vals + [np.full(g + 1, np.nan)])
        self.g = g
        self.T = np.array(self.tiles, SP_TILE)
        rec = lambda lst, dt: np.array(lst, dt) if lst else np.zeros(1, dt)
        self.A, self.S, self.B = rec(self.aslots, SP_ASLOT), rec(self.sslots, SP_SSLOT), rec(self.bslots, SP_BSLOT)
        return self

    def run(self, dc, max_nR, tiles=None):
        T = self.T if tiles is None else tiles
        Y = np.empty_like(self.X)
        Y.view(np.uint64)[:] = SENT
        dc.ok("dc_spmm", T if len(T) else np.zeros(1, SP_TILE), len(T), self.A, len(self.aslots), self.S, len(self.sslots), self.B, len(self.bslots), self.g,
              self.X, self.X.size, Y, Y.size, self.I, self.I.size, self.V, self.V.size, max_nR)
        return Y

    def owned(self, tiles=None):
        """mask of the Y elements the tiles write"""
        m = np.zeros(self.X.size, bool)
        for t in (self.T if tiles is None else tiles):
            o = self.g + int(t["off"])
            m[o:o + int(t["nrows"]) * int(t["nR"])] = True
        return m

    def check(self, Y, what, tiles=None):
        g = self.g
        x = self.X[g:-g].astype(LD)
        I, V = self.I[g:], self.V[g:]
        assert (bits(Y[~self.owned(tiles)]) == SENT).all(), "%s: Y written outside the rows of its tiles" % what
        for ti, t in enumerate(self.T if tiles is None else tiles):
            nR, nrows, off = int(t["nR"]), int(t["nrows"]), int(t["off"])
            c = np.arange(nR)
            ref = np.zeros((nrows, nR), LD)
            ab = np.zeros((nrows, nR), LD)
            a = self.A[t["a_begin"]:t["a_begin"] + t["a_count"]]
            if len(a):
                terms = a["w"][:, :nrows, None].astype(LD) * x[a["src"][:, :nrows, None] + c]
                ref += terms.sum(0); ab += np.abs(terms).sum(0)
            s = self.S[t["s_begin"]:t["s_begin"] + t["s_count"]]
            if len(s):
                terms = s["w"][:, :nrows, None].astype(LD) * x[off + s["roff"][:, :nrows, None].astype(np.int64) + c]
                ref += terms.sum(0); ab += np.abs(terms).sum(0)
            nterms = len(a) + len(s)
            for b in self.B[t["b_begin"]:t["b_begin"] + t["b_count"]]:
                W, ld = int(b["W"]), int(b["ld"])
                if W == 0:
                    continue
                e = (np.arange(W)[:, None] * ld + c).ravel()
                cols = I[int(b["ecol"]) + e].reshape(W, nR).astype(np.int64)
                vals = V[int(b["eval"]) + e].reshape(W, nR).astype(LD)
                base = (off + b["roff"][:nrows].astype(np.int64)) if b["all_in"] else b["src"][:nrows]
                terms = b["w"][:nrows, None, None].astype(LD) * vals[None] * x[base[:, None, None] + cols[None]]
                ref += terms.sum(1); ab += np.abs(terms).sum(1)
                nterms += 2 * W
            got = Y[g + off:g + off + nrows * nR].reshape(nrows, nR)
            assert_bound(got, ref, ab, nterms, "%s: tile %d (nR %d, nrows %d, off %s)" % (what, ti, nR, nrows, "odd" if off & 1 else "even"))


def _max_nr(mode, widest):
    return [widest, min(SP_MAX_NR, widest + 1 + widest // 3), SP_MAX_NR][mode]


@pytest.mark.parametrize("nR", NRS)
def test_spmm_tile_shapes(dc, nR):
    """one launch of 8 tiles of width nR: nrows 1-4 at even and odd offsets, slot counts cycling through both sides of
    the a-/s-slot batch of 24 and the b-slot batch of 8, W 0/1/5, ld = nR, rounded up to 32 and larger, all_in and L2
    b-slots alternating; max_nR the tile width, above it or SP_MAX_NR by turns"""
    k = NRS.index(nR)
    rng = rng_for("spmm-shapes", nR)
    max_nR = _max_nr(k % 3, nR)
    plan = SpPlan(rng)
    for i in range(8):
        plan.tile(nR, i % 4 + 1, (i // 4 + k) % 2, SLOT_COUNTS[(i + k) % 7], SLOT_COUNTS[(i + 2 * k + 3) % 7], BSLOT_COUNTS[(i + 3 * k + 5) % 7],
                  ld_mode=i + k, all_in_first=i)
    plan.finish(guard_for(SP_ROWS * max_nR))
    Y = plan.run(dc, max_nR)
    plan.check(Y, "nR %d max_nR %d" % (nR, max_nR))
    assert (bits(plan.run(dc, max_nR)) == bits(Y)).all(), "two calls differ"


def test_spmm_large_batch_order_and_isolation(dc):
    """640 tiles of mixed width in one launch; the same tiles reversed and shuffled give the same bits, and so does each
    of a few tiles launched alone"""
    rng = rng_for("spmm-batch")
    plan = SpPlan(rng)
    wp = 1.0 / np.sqrt(np.array(NRS, float))
    for i in range(640):
        nR = int(rng.choice(NRS, p=wp / wp.sum()))
        small = [0, 1, 2, 5, 23, 24, 25]
        plan.tile(nR, int(rng.integers(1, SP_ROWS + 1)), int(rng.integers(2)), int(rng.choice(small)), int(rng.choice(small)),
                  int(rng.choice([0, 1, 2, 3, 8, 9])), ld_mode=i, all_in_first=i)
    plan.finish(guard_for(SP_ROWS * SP_MAX_NR))
    Y = plan.run(dc, SP_MAX_NR)
    plan.check(Y, "batch of 640")
    for name, order in (("reversed", np.arange(len(plan.T))[::-1]), ("shuffled", rng.permutation(len(plan.T)))):
        assert (bits(plan.run(dc, SP_MAX_NR, plan.T[order])) == bits(Y)).all(), "tile order %s changes bits" % name
    widest = int(np.argmax(plan.T["nR"]))
    partial = int(np.flatnonzero(plan.T["nrows"] < SP_ROWS)[0])
    for i in sorted({0, len(plan.T) - 1, widest, partial, *rng.choice(len(plan.T), 3, replace=False).tolist()}):
        one = plan.T[i:i + 1]
        Yi = plan.run(dc, SP_MAX_NR, one)
        m = plan.owned(one)
        assert (bits(Yi[m]) == bits(Y[m])).all(), "tile %d alone differs from the batch" % i
        assert (bits(Yi[~m]) == SENT).all(), "tile %d alone wrote outside its rows" % i


def test_spmm_no_tiles_leaves_y(dc):
    plan = SpPlan(rng_for("spmm-empty"))
    plan.tile(33, 3, 1, 2, 2, 2)
    plan.finish(guard_for(SP_ROWS * 33))
    Y = plan.run(dc, 33, plan.T[:0])
    assert (bits(Y) == SENT).all()


def test_spmm_plan_validation(dc):
    """the shim refuses, before any launch, plans that would reach outside a buffer through the rows past a partial
    tile, an in-tile offset or a gathered column, and a Y guard that cannot hold SP_ROWS rows of max_nR"""
    def fresh():
        plan = SpPlan(rng_for("spmm-refuse"))
        plan.tile(40, 2, 0, 1, 1, 2, ld_mode=1, all_in_first=0)      # b-slot 0: L2, W = 1; b-slot 1: all_in, W = 5
        return plan.finish(guard_for(SP_ROWS * 64))
    plan = fresh()
    plan.run(dc, 64)
    cases = {
        "a-slot source row": lambda p: p.A[0]["src"].__setitem__(3, p.X.size - 2 * p.g - 10),          # row 3 >= nrows
        "s-slot source row": lambda p: p.S[0]["roff"].__setitem__(1, 2 * 40 - 39),                        # row 1 < nrows: past the tile
        "all_in gather": lambda p: p.I.__setitem__(p.g + int(p.B[1]["ecol"]), 10 ** 6),
        "b-slot gather": lambda p: p.B[0]["src"].__setitem__(2, p.X.size),
    }
    for what, spoil in cases.items():
        p = fresh()
        spoil(p)
        Y = np.empty_like(p.X)
        msg = dc.refused("dc_spmm", p.T, 1, p.A, 1, p.S, 1, p.B, 2, p.g, p.X, p.X.size, Y, Y.size, p.I, p.I.size, p.V, p.V.size, 64)
        assert what in msg, (what, msg)
    p = fresh()
    Y = np.empty_like(p.X)
    assert "guard" in dc.refused("dc_spmm", p.T, 1, p.A, 1, p.S, 1, p.B, 2, p.g, p.X, p.X.size, Y, Y.size, p.I, p.I.size, p.V, p.V.size, p.g // SP_ROWS + 1)


# ---------------------------------------------------------------------------------------------------------------------
#  syevd_batch
# ---------------------------------------------------------------------------------------------------------------------
SIZES = [1, 2, 63, 64, 65, 127, 128, 129, 192, 193]
CUDA_SIZES = [257, 512, 832]
C_EIG = 32.0
TAU_W, TAU_O = 5e-14, 1e-12   # the caps: test_gpu_parity.py's fixed eigensolver tolerances
EG = 512   # guard between payloads (4 KiB)


def _sizes(dc):
    return SIZES + (CUDA_SIZES if dc.name == "cuda" else [])


def syevd(dc, mats, rng):
    """one dc_syevd call over mats placed in a shuffled order at random parities; returns [(w, V)], after checking the
    guards and that a second call gives the same bits"""
    nb = len(mats)
    n = np.array([m.shape[0] for m in mats], np.int32)
    a_off, w_off = np.zeros(nb, np.int64), np.zeros(nb, np.int64)
    na = nw = 0
    for b in rng.permutation(nb):
        na += EG + int((na + EG) % 2 != rng.integers(2)); a_off[b] = na; na += int(n[b]) ** 2
        nw += EG + int((nw + EG) % 2 != rng.integers(2)); w_off[b] = nw; nw += int(n[b])
    A0 = np.empty(na + EG); A0.view(np.uint64)[:] = SENT
    W0 = np.empty(nw + EG); W0.view(np.uint64)[:] = SENT
    for b, m in enumerate(mats):
        A0[a_off[b]:a_off[b] + n[b] ** 2] = m.ravel()
    outs = []
    for _ in range(2):
        A, W = A0.copy(), W0.copy()
        dc.ok("dc_syevd", nb, n, a_off, w_off, A, A.size, W, W.size, EG)
        outs.append((A, W))
    (A, W), (A2, W2) = outs
    assert (bits(A) == bits(A2)).all() and (bits(W) == bits(W2)).all(), "two calls differ"
    ma, mw = np.ones(A.size, bool), np.ones(W.size, bool)
    for b in range(nb):
        ma[a_off[b]:a_off[b] + n[b] ** 2] = False
        mw[w_off[b]:w_off[b] + n[b]] = False
    assert (bits(A[ma]) == SENT).all() and (bits(W[mw]) == SENT).all(), "a guard between payloads changed"
    return [(W[w_off[b]:w_off[b] + n[b]].copy(), A[a_off[b]:a_off[b] + n[b] ** 2].reshape(n[b], n[b]).copy()) for b in range(nb)]


def check_eig(w, V, R, what):
    n = len(w)
    ref = np.linalg.eigvalsh(R)
    nrm = float(np.abs(ref).max())
    assert np.all(np.diff(w) >= 0), "%s: eigenvalues not ascending" % what
    Vl, Rl = V.astype(LD), R.astype(LD)
    res = np.sqrt((((Rl @ Vl.T) - Vl.T * w.astype(LD)[None, :]) ** 2).sum(0)).max()
    orth = np.abs(Vl @ Vl.T - np.eye(n, dtype=LD)).max()
    for name, got, bound in (("eigenvalue error", np.abs(w - ref).max(), min(C_EIG * n * U, TAU_W) * nrm),
                             ("orthogonality", float(orth), min(C_EIG * n * U, TAU_O)),
                             ("residual", float(res), C_EIG * n * U * nrm)):
        assert got <= bound, "%s: %s %.3g > %.3g" % (what, name, got, bound)


def _multiplet(rng, n):
    lam = np.concatenate([np.full(m, v) for m, v in zip(np.resize(np.arange(2, 9), n), np.exp(-rng.uniform(0, 20, n)))])[:n]
    return with_spectrum(rng, np.sort(lam)[::-1])


FAMILIES = {
    "rho": rho_like,
    "multiplets": _multiplet,
    "zero": lambda rng, n: np.zeros((n, n)),
    "indefinite": lambda rng, n: with_spectrum(rng, rng.standard_normal(n)),
    "negative-definite": lambda rng, n: -rho_like(rng, n) - 0.1 * np.eye(n),
}


@pytest.mark.parametrize("family", list(FAMILIES))
def test_syevd_families(dc, family):
    rng = rng_for("syevd", family)
    mats = [FAMILIES[family](rng, n) for n in _sizes(dc)]
    for (w, V), R in zip(syevd(dc, mats, rng), mats):
        check_eig(w, V, R, "%s n %d" % (family, len(w)))


def test_syevd_diagonal_is_exact(dc):
    """no rotation on either path: w = sort(diag), row k = e_argsort(diag)[k] (stable on the many ties), bit for bit"""
    rng = rng_for("syevd-diag")
    diags = [rng.integers(-3, 4, n) * 0.5 + (rng.integers(0, 3, n) == 0) * rng.standard_normal(n) for n in _sizes(dc)]
    diags = [np.where(d == 0, 0.0, d) for d in diags]          # +0 only: a sum of ±0 products gives +0
    for (w, V), d in zip(syevd(dc, [np.diag(d) for d in diags], rng), diags):
        o = np.argsort(d, kind="stable")
        assert (bits(w) == bits(d[o])).all(), "n %d: eigenvalues" % len(d)
        assert (bits(V) == bits(np.eye(len(d))[o])).all(), "n %d: eigenvectors" % len(d)


def _graded(rng, n, m):
    """A = Q Λ Qᵀ in longdouble (Q a product of three Householder reflections), spectrum 1 .. 1e-5 on the top m states and
    1e-7 .. 1e-14 below: returns A rounded to float64, the exact top-m projector and the gap"""
    lam = np.concatenate([np.logspace(0, -5, m), np.logspace(-7, -14, n - m)]).astype(LD)
    Q = np.eye(n, dtype=LD)
    for _ in range(3):
        v = rng.standard_normal(n).astype(LD)
        Q = Q - (2 / (v @ v)) * np.outer(Q @ v, v)
    A = (Q * lam[None, :]) @ Q.T
    Qm = Q[:, :m]
    return np.asarray(A, np.float64), Qm @ Qm.T, float(lam[m - 1] - lam[m])


@pytest.mark.parametrize("n,m", [(48, 17), (64, 40), (129, 50), (193, 96)])
def test_syevd_graded_subspace(dc, n, m):
    """the subspace the truncation keeps: the projector onto the m largest eigenvectors against the exact one"""
    rng = rng_for("syevd-graded", n, m)
    A, P, gap = _graded(rng, n, m)
    (w, V), = syevd(dc, [A], rng)
    check_eig(w, V, A, "graded n %d" % n)
    Vm = V[n - m:].astype(LD)
    err = np.linalg.norm(np.asarray(Vm.T @ Vm - P, np.float64), 2)
    bound = C_EIG * n * U * float(np.abs(w).max()) / gap
    assert err <= bound, "graded n %d m %d: projector error %.3g > %.3g" % (n, m, err, bound)


def test_syevd_mixed_batch(dc):
    """≥ 40 blocks of both paths in one call, sizes shuffled, every block with its own spectrum (shifted by its index):
    a result written to another block fails its eigenvalues"""
    rng = rng_for("syevd-mixed")
    sizes = [1, 2, 3, 17, 33, 63, 64, 64, 65, 65, 66, 96, 127, 128, 129, 130, 160, 192, 193] + [int(s) for s in rng.integers(1, 140, 24)]
    if dc.name == "cuda":
        sizes += [257, 300]
    sizes = [sizes[i] for i in rng.permutation(len(sizes))]
    mats = [with_spectrum(rng, b + 0.25 + 0.5 * rng.random(n)) for b, n in enumerate(sizes)]
    for b, ((w, V), R) in enumerate(zip(syevd(dc, mats, rng), mats)):
        assert b <= w.min() and w.max() <= b + 1, "block %d: spectrum of another block" % b
        check_eig(w, V, R, "mixed block %d n %d" % (b, len(w)))
