"""Kernel-by-kernel tests of the device layer (csrc/dev.h): chain_kernel / reduce_kernel, gram, the Gram-Schmidt and Ritz
kernels of the eigensolver, lanczos_batch and the streaming kernels, each called directly through the test-only shim
tests/devcheck/devcheck.cpp at the shapes where the kernels branch: every tile extent class of chain_kernel's dispatch,
every K tail, both copy-ring depths, every template instance of gs_pass / gs_final, the block-count edges of the
reductions.  Every test runs on two backends with the same cases and tolerances: `host` (the shim over the host
emulation tests/plancheck/dev_host*.cpp; proves the harness and the references without a GPU) and `cuda` (the shim over
the product's own sm_100a object; marked gpu).

Guard bands.  Every buffer handed to the shim carries a guard of at least 4 KiB and one leading dimension on each side.
Operand guards and padding (rows [n, ld), rows past a tile, vectors past nvec) hold NaN, so an over-read turns a result
NaN; output guards and untouched gaps (ldc padding, elements between tiles) hold a sentinel bit pattern that must survive.

Reference and tolerance.  Every reference is computed in NumPy np.longdouble (the 80-bit x87 format on x86-64, a 64-bit
significand), independently of the emulation's loops.  An element that is a sum of N rounded float64 products, N counted
over the whole chain of that element including coefficient multiplies and the additions of a part reduction, must satisfy

    |got - ref| <= (N + 2) · 2^-53 · Σ|terms|.

This is the classical a-priori bound of floating-point summation (Higham, Accuracy and Stability of Numerical Algorithms,
2nd ed., §3.1 and §4.2) plus the rounding of the products: it holds for any summation order and any mix of separate and
fused multiply-adds, so it covers DMMA's fused steps, any reduction tree and the compiler's contractions; the longdouble
reference adds ~2^-64 relative.  It still has teeth: one dropped, duplicated or mis-strided product moves an element by
about one term, ~Σ|terms|/N, which is 2^53/(N(N+2)) times the bound.  In the chain tests N <= ~1000, a factor of at least
9·10^9; in the reductions at n = 10^6 a single lost element is 9·10^3 times the bound, and what those kernels lose when
they are wrong (a block, a warp, a grid-stride pass: 256 elements or more) at least 2·10^6 times.  Where dev.h promises
bit-reproducibility (two calls, the two ring depths, a Lanczos column alone or in a batch) bit equality is asserted, and
where the data are exact (dyadic Gram inputs, copies, splitmix64) exact equality.
"""
import ctypes as C

import numpy as np
import pytest

from devcheck_common import (LD, SENT, SP_ASLOT, SP_BSLOT, SP_MAX_NR, SP_ROWS, SP_SSLOT, SP_TILE, U, Backend, assert_bound, assert_guards,
                             assert_unchanged, bits, guard_for, lib_path, rng_for, sentinel, wrap)

DEEP_BELOW = 1800                        # run_chain: launches below this many items take the three-stage copy ring
RED_BLOCKS = 592                         # grid of the streaming kernels
MAX_BASIS = 39
SEG_GEMM, SEG_AXPY, SEG_DIAG, SEG_CSRA, SEG_CSRB, SEG_CSRADD = range(6)
SEGF_A_X, SEGF_B_X = 1, 2

SEG = np.dtype([("A", "<i8"), ("B", "<i8"), ("rowptr", "<i8"), ("colidx", "<i8"), ("lda_m", "<i8"), ("lda_k", "<i8"), ("ldb_n", "<i8"),
                ("ldb_k", "<i8"), ("coef", "<f8"), ("K", "<i4"), ("type", "<i4"), ("row0", "<i4"), ("d", "<i4"), ("flags", "<i4"), ("pad", "<i4")])
ITEM = np.dtype([("C", "<i8"), ("ldc", "<i8"), ("m0", "<i4"), ("n0", "<i4"), ("tm", "<i4"), ("tn", "<i4"), ("seg_begin", "<i4"), ("seg_end", "<i4"),
                 ("mode", "<i4"), ("c_in_y", "<i4")])
RED = np.dtype([("dst", "<i8"), ("ldc", "<i8"), ("src_off", "<i8"), ("tm", "<i4"), ("tn", "<i4"), ("nparts", "<i4"), ("dst_in_y", "<i4")])
assert SEG.itemsize == 96 and ITEM.itemsize == 48 and RED.itemsize == 40

EXTS = [1, 8, 9, 16, 17, 24, 31, 32, 33, 40, 48, 49, 56, 63, 64]
KS = [0, 1, 3, 4, 5, 8, 9, 12, 13, 15, 16, 17, 31, 32, 33, 48, 200, 1000]
COEFS = [1.0, -0.5, 1.0 / 3.0]
CELL = 80   # rows / columns of the operand cells the work items cut their tiles from


# ---------------------------------------------------------------------------------------------------------------------
#  backend and buffers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["host", pytest.param("cuda", marks=pytest.mark.gpu)])
def dc(request):
    # the int arguments of every dc_* entry point are declared long long or int; ctypes passes c_longlong, which is
    # also right for int arguments on x86-64 / aarch64 (registers and 8-byte stack slots)
    return Backend(request.param, lib_path(request.param))


# ---------------------------------------------------------------------------------------------------------------------
#  run_chain / run_reduce
# ---------------------------------------------------------------------------------------------------------------------
def store(M, lm, lk):
    """a logical R×K matrix at element strides (lm, lk), NaN wherever the matrix has no element"""
    R, K = M.shape
    buf = np.full(max(1, (R - 1) * lm + (K - 1) * lk + 1) if R and K else 1, np.nan)
    if R and K:
        buf[(np.arange(R)[:, None] * lm + np.arange(K)[None, :] * lk).ravel()] = M.ravel()
    return buf


class Pool:
    """a growing host buffer of doubles (or ints); put() returns the element offset of the stored block"""

    def __init__(self, dtype=np.float64, fill=np.nan):
        self.parts, self.n, self.dtype, self.fill = [], 0, dtype, fill

    def put(self, arr, odd=False):
        arr = np.asarray(arr, self.dtype).ravel()
        if odd != bool(self.n & 1):       # 8-byte but not 16-byte aligned when odd
            self.parts.append(np.full(1, self.fill, self.dtype)); self.n += 1
        off = self.n
        self.parts.append(arr); self.n += arr.size
        return off

    def array(self):
        return np.concatenate(self.parts + [np.full(1, self.fill, self.dtype)]) if self.parts else np.full(1, self.fill, self.dtype)


class OutPool:
    """an output pool (O, y or w): sentinel everywhere except the preset values of accumulate tiles"""

    def __init__(self):
        self.n = 0
        self.preset = []

    def tile(self, tm, tn, ldc, init=None):
        off = self.n + 1    # one sentinel between tiles
        self.n = off + (tm - 1) * ldc + tn + (ldc - tn)
        if init is not None:
            self.preset.append((off, ldc, init))
        return off

    def array(self, g):
        full = sentinel(self.n + 1, g)
        for off, ldc, init in self.preset:
            tm, tn = init.shape
            full[g + off + (np.arange(tm)[:, None] * ldc + np.arange(tn)[None, :])] = init
        return full


LAYOUTS = {"mk,nk": (True, True), "mk,kn": (True, False), "km,nk": (False, True), "km,kn": (False, False)}


class Operands:
    """Stored operand pairs (A: CELL×K, B: K×CELL logical) in a pool, each product computed once in longdouble: the
    work items slice it.  layout: A contiguous along k (mk) or m (km), B along k (nk) or n (kn); 'strided': neither."""

    def __init__(self, rng):
        self.rng = rng
        self.cache = {}

    def get(self, pool, layout, K, in_x=False):
        key = (id(pool), layout, K, in_x)
        if key in self.cache:
            return self.cache[key]
        A = self.rng.standard_normal((CELL, K))
        B = self.rng.standard_normal((K, CELL))
        if layout == "strided":
            lda_m, lda_k, ldb_n, ldb_k = 2 * K + 3, 2, 3, 3 * CELL + 1
        else:
            a_mk, b_nk = LAYOUTS[layout]
            lda_m, lda_k = ((K + 3) | 1, 1) if a_mk else (1, CELL + 3)
            ldb_n, ldb_k = ((K + 2) | 1, 1) if b_nk else (1, CELL + 1)
        offA = pool.put(store(A, lda_m, lda_k), odd=True)
        offB = pool.put(store(B.T, ldb_n, ldb_k), odd=True)     # B(k, n) at n·ldb_n + k·ldb_k
        prod = A.astype(LD) @ B.astype(LD)
        absp = np.abs(A).astype(LD) @ np.abs(B).astype(LD)
        r = dict(A=offA, B=offB, lda_m=lda_m, lda_k=lda_k, ldb_n=ldb_n, ldb_k=ldb_k, K=K, prod=prod, absp=absp)
        self.cache[key] = r
        return r


def seg_record(**kw):
    s = np.zeros(1, SEG)[0]
    for k, v in kw.items():
        s[k] = v
    return s


class ChainPlan:
    def __init__(self):
        self.D, self.X, self.I = Pool(), Pool(), Pool(np.int32, 0)
        self.O, self.Y, self.W = OutPool(), OutPool(), OutPool()
        self.segs, self.items, self.red = [], [], []
        self.expect = []      # (pool name, offset, ldc, ref, absref, N, init)

    def pool(self, name):
        return {"O": self.O, "Y": self.Y, "W": self.W}[name]

    def item(self, segs, m0, n0, tm, tn, ref, absref, N, where="O", mode=0, ldc=None, init=None, expect=True):
        ldc = tn + 3 if ldc is None else ldc
        off = self.pool(where).tile(tm, tn, ldc, init if mode == 1 else None)
        b = len(self.segs)
        self.segs.extend(segs)
        it = np.zeros(1, ITEM)[0]
        it["C"] = off if where == "O" else 8 * off
        it["ldc"], it["m0"], it["n0"], it["tm"], it["tn"] = ldc, m0, n0, tm, tn
        it["seg_begin"], it["seg_end"], it["mode"], it["c_in_y"] = b, len(self.segs), mode, {"O": 0, "Y": 1, "W": 2}[where]
        self.items.append(it)
        if expect:
            self.expect.append((where, off, ldc, ref, absref, N, init if mode == 1 else None))
        return off

    def arrays(self, items=None):
        items = self.items if items is None else items
        g = guard_for()
        return dict(items=np.array(items, ITEM), segs=np.array(self.segs if self.segs else [seg_record()], SEG),
                    red=np.array(self.red if self.red else [np.zeros(1, RED)[0]], RED), g=g,
                    D=wrap(self.D.array(), g), I=wrap(self.I.array(), g, "nan"), X=wrap(self.X.array(), g),
                    O=self.O.array(g), Y=self.Y.array(g), W=self.W.array(g))

    def run(self, dc, items=None):
        a = self.arrays(items)
        nred = len(self.red)
        dc.ok("dc_chain", a["items"], len(a["items"]), a["segs"], len(self.segs), a["red"], nred, a["g"], a["D"], a["D"].size,
              a["I"], a["I"].size, a["X"], a["X"].size, a["Y"], a["Y"].size, a["W"], a["W"].size, a["O"], a["O"].size)
        return a

    def check(self, a, expect=None):
        g = a["g"]
        written = {k: np.zeros(a[k].size - 2 * g, bool) for k in "OYW"}
        for where, off, ldc, ref, absref, N, init in (self.expect if expect is None else expect):
            tm, tn = ref.shape
            idx = off + np.arange(tm)[:, None] * ldc + np.arange(tn)[None, :]
            got = a[where][g:-g][idx]
            r, ab = ref, absref
            if init is not None:
                r, ab, N = ref + init.astype(LD), absref + np.abs(init).astype(LD), np.asarray(N) + 1
            assert_bound(got, r, ab, N, "%s tile at %d (%dx%d)" % (where, off, tm, tn))
            written[where][idx] = True
        for k in "OYW":
            assert_guards(a[k], g, k)
            body = a[k][g:-g]
            assert (bits(body[~written[k]]) == SENT).all(), "%s: an element outside every tile was written" % k


def grid_plan():
    """Every tile extent pair of EXTS in each of the four DMMA layouts, K and the coefficient cycling; the full 64×64
    tile with every K and every coefficient (the four K-tail bodies at coefficient 1, the generic body otherwise)."""
    plan = ChainPlan()
    ops = Operands(rng_for("grid"))
    for li, layout in enumerate(LAYOUTS):
        cases = [(tm, tn, KS[(7 * idx + 5 * li) % len(KS)], COEFS[(idx + li) % 3], (0, 3, 16)[idx % 3], (16, 0, 5)[idx % 3])
                 for idx, (tm, tn) in enumerate((tm, tn) for tm in EXTS for tn in EXTS)]
        cases += [(64, 64, K, c, 16 * (j & 1), 7 * (j % 3 == 2)) for j, (K, c) in enumerate((K, c) for K in KS for c in COEFS)]
        for tm, tn, K, coef, m0, n0 in cases:
            op = ops.get(plan.D, layout, K)
            s = seg_record(A=op["A"], B=op["B"], lda_m=op["lda_m"], lda_k=op["lda_k"], ldb_n=op["ldb_n"], ldb_k=op["ldb_k"], coef=coef, K=K,
                           type=SEG_GEMM)
            ref = LD(coef) * op["prod"][m0:m0 + tm, n0:n0 + tn]
            absref = LD(abs(coef)) * op["absp"][m0:m0 + tm, n0:n0 + tn]
            plan.item([s], m0, n0, tm, tn, ref, absref, K + 1)
    return plan


def padded(plan, n_total):
    """the plan's items plus copies of them, writing to tiles of their own, up to n_total items (the two-stage ring)"""
    items = list(plan.items)
    extra = []
    k = 0
    while len(items) < n_total:
        src, (where, off, ldc, ref, absref, N, init) = plan.items[k], plan.expect[k]
        it = src.copy()
        tm, tn = int(it["tm"]), int(it["tn"])
        noff = plan.O.tile(tm, tn, ldc, init)
        it["C"], it["c_in_y"] = noff, 0
        items.append(it)
        extra.append(("O", noff, ldc, ref, absref, N, init))
        k += 1
    return items, extra


def chain_tile(a, where, off, ldc, tm, tn):
    g = a["g"]
    return a[where][g:-g][off + np.arange(tm)[:, None] * ldc + np.arange(tn)[None, :]]


def test_chain_gemm_tiles_k_tails_layouts_and_ring_depths(dc):
    """chain_kernel on single-GEMM chains: all 225 tile extent pairs in each layout (every per-warp fragment class of the
    dispatch, including warps that own none), every K of KS, three coefficients, odd leading dimensions with NaN padding,
    operands 8- but not 16-byte aligned.  The same items in a launch below 1800 items (three-stage ring) and padded above
    it (two-stage ring) must give the same bits, and two runs of one launch too."""
    plan = grid_plan()
    assert len(plan.items) < DEEP_BELOW
    a1 = plan.run(dc)
    plan.check(a1)
    a2 = plan.run(dc)
    for k in "OYW":
        assert (bits(a1[k]) == bits(a2[k])).all(), "two runs of one launch differ"
    items, extra = padded(plan, DEEP_BELOW + 7)
    a3 = plan.run(dc, items)
    plan.check(a3, plan.expect + extra)
    for (where, off, ldc, ref, _, _, _), (w2, off2, _, _, _, _, _) in zip(plan.expect, extra):
        t1 = chain_tile(a1, where, off, ldc, *ref.shape)
        assert (bits(t1) == bits(chain_tile(a3, where, off, ldc, *ref.shape))).all(), "the ring depth changed the arithmetic"
        assert (bits(t1) == bits(chain_tile(a3, w2, off2, ldc, *ref.shape))).all(), "a copy of an item in one launch differs"


class Sparse:
    """a CSR matrix of 120 rows × 96 columns with empty rows, short rows and rows longer than a tile"""

    def __init__(self, rng, plan, vals_in_x):
        nrows, ncols = 120, 96
        lens = rng.choice([0, 0, 1, 3, 5, 70], size=nrows)
        rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
        cols = np.concatenate([rng.choice(ncols, size=L, replace=L > ncols) for L in lens]).astype(np.int32) if lens.sum() else np.zeros(0, np.int32)
        vals = rng.standard_normal(cols.size)
        self.dense = np.zeros((nrows, ncols), LD)
        self.absd = np.zeros((nrows, ncols), LD)
        self.cnt = lens
        r_of = np.repeat(np.arange(nrows), lens)
        np.add.at(self.dense, (r_of, cols), vals.astype(LD))
        np.add.at(self.absd, (r_of, cols), np.abs(vals).astype(LD))
        self.rowptr = plan.I.put(rowptr)
        self.colidx = plan.I.put(cols if cols.size else np.zeros(1, np.int32))
        self.vals_in_x = vals_in_x
        pool = plan.X if vals_in_x else plan.D
        off = pool.put(vals if vals.size else np.zeros(1), odd=True)
        self.vals = 8 * off if vals_in_x else off
        self.ncols = ncols


def mixed_plan(seed):
    """Chains of 1-12 segments on ragged and full tiles mixing every segment type: GEMMs of all layouts (and a strided one)
    with K = 0 among them, AXPY with lda_k != 1, DIAG and CSRADD with negative and positive offsets, CSRA / CSRB with
    row0 != 0, empty rows and rows longer than a tile, operands in x (SEGF_A_X / SEGF_B_X); outputs plain, in y (c_in_y 1)
    and in w (c_in_y 2), stored or accumulated; partial tiles in w summed by run_reduce (1-5 parts) into y and into a
    plain pointer."""
    rng = rng_for("mixed", seed)
    plan = ChainPlan()
    ops = Operands(rng)
    sparse = [Sparse(rng, plan, False), Sparse(rng, plan, True)]
    # dense factors of the sparse segments: CSRA's right factor X(k, n) (96 × CELL), CSRB's left factor A(m, k) (CELL × 96)
    Fr = rng.standard_normal((96, CELL)); Fl = rng.standard_normal((CELL, 96)); Ax = rng.standard_normal((CELL, CELL))
    fr = [dict(off=plan.D.put(store(Fr, CELL + 1, 1), odd=True), x=False, ldb_k=CELL + 1, ldb_n=1),
          dict(off=8 * plan.X.put(store(Fr, 1, 97), odd=True), x=True, ldb_k=1, ldb_n=97)]
    fl = [dict(off=plan.D.put(store(Fl, 1, CELL + 3), odd=True), x=False, lda_m=1, lda_k=CELL + 3),
          dict(off=8 * plan.X.put(store(Fl, 99, 1), odd=True), x=True, lda_m=99, lda_k=1)]
    ax = [dict(off=plan.D.put(store(Ax, 1, CELL + 5), odd=True), x=False, lda_m=1, lda_k=CELL + 5),
          dict(off=8 * plan.X.put(store(Ax, 2 * CELL + 1, 2), odd=True), x=True, lda_m=2 * CELL + 1, lda_k=2)]
    layouts = list(LAYOUTS) + ["strided"]
    kmix = [0, 1, 3, 5, 9, 13, 16, 17, 33, 48, 200]

    def chain(m0, n0, tm, tn, nseg):
        segs = []
        ref = np.zeros((tm, tn), LD); absref = np.zeros((tm, tn), LD); N = 0
        rows, cols = slice(m0, m0 + tm), slice(n0, n0 + tn)
        for _ in range(nseg):
            typ = rng.choice(6, p=[0.35, 0.13, 0.13, 0.13, 0.13, 0.13])
            coef = COEFS[rng.integers(3)]
            if typ == SEG_GEMM:
                in_x = bool(rng.integers(2))
                op = ops.get(plan.X if in_x else plan.D, layouts[rng.integers(len(layouts))], int(rng.choice(kmix)), in_x)
                fl_ = SEGF_A_X | SEGF_B_X if in_x else 0
                A, B = (8 * op["A"], 8 * op["B"]) if in_x else (op["A"], op["B"])
                segs.append(seg_record(A=A, B=B, lda_m=op["lda_m"], lda_k=op["lda_k"], ldb_n=op["ldb_n"], ldb_k=op["ldb_k"], coef=coef, K=op["K"],
                                       type=SEG_GEMM, flags=fl_))
                ref += LD(coef) * op["prod"][rows, cols]; absref += LD(abs(coef)) * op["absp"][rows, cols]; N += op["K"] + 1
            elif typ == SEG_AXPY:
                f = ax[rng.integers(2)]
                segs.append(seg_record(A=f["off"], lda_m=f["lda_m"], lda_k=f["lda_k"], coef=coef, type=SEG_AXPY, flags=SEGF_A_X if f["x"] else 0))
                ref += LD(coef) * Ax[rows, cols].astype(LD); absref += LD(abs(coef)) * np.abs(Ax[rows, cols]).astype(LD); N += 1
            elif typ == SEG_DIAG:
                d = int(rng.choice([-20, -9, -1, 0, 1, 5, 17]))
                segs.append(seg_record(coef=coef, type=SEG_DIAG, d=d))
                e = ((np.arange(m0, m0 + tm)[:, None] + d) == np.arange(n0, n0 + tn)[None, :]).astype(LD)
                ref += LD(coef) * e; absref += LD(abs(coef)) * e; N += 1
            else:
                sp = sparse[rng.integers(2)]
                row0 = int(rng.choice([0, 7, 30]))
                bflag = SEGF_B_X if sp.vals_in_x else 0
                if typ == SEG_CSRA:
                    f = fr[rng.integers(2)]
                    S, Sa = sp.dense[row0 + m0:row0 + m0 + tm], sp.absd[row0 + m0:row0 + m0 + tm]
                    segs.append(seg_record(A=f["off"], B=sp.vals, rowptr=sp.rowptr, colidx=sp.colidx, ldb_n=f["ldb_n"], ldb_k=f["ldb_k"], coef=coef,
                                           type=SEG_CSRA, row0=row0, flags=bflag | (SEGF_A_X if f["x"] else 0)))
                    ref += LD(coef) * (S @ Fr[:, cols].astype(LD)); absref += LD(abs(coef)) * (Sa @ np.abs(Fr[:, cols]).astype(LD))
                    N += int(sp.cnt[row0 + m0:row0 + m0 + tm].max()) + 1
                elif typ == SEG_CSRB:
                    f = fl[rng.integers(2)]
                    S, Sa = sp.dense[row0 + n0:row0 + n0 + tn], sp.absd[row0 + n0:row0 + n0 + tn]
                    segs.append(seg_record(A=f["off"], B=sp.vals, rowptr=sp.rowptr, colidx=sp.colidx, lda_m=f["lda_m"], lda_k=f["lda_k"], coef=coef,
                                           type=SEG_CSRB, row0=row0, flags=bflag | (SEGF_A_X if f["x"] else 0)))
                    ref += LD(coef) * (Fl[rows].astype(LD) @ S.T); absref += LD(abs(coef)) * (np.abs(Fl[rows]).astype(LD) @ Sa.T)
                    N += int(sp.cnt[row0 + n0:row0 + n0 + tn].max()) + 1
                else:
                    d = int(rng.choice([-6, -1, 0, 2, 11]))
                    segs.append(seg_record(B=sp.vals, rowptr=sp.rowptr, colidx=sp.colidx, coef=coef, type=SEG_CSRADD, row0=row0, d=d, flags=bflag))
                    S, Sa = sp.dense[row0 + m0:row0 + m0 + tm], sp.absd[row0 + m0:row0 + m0 + tm]
                    c = np.arange(n0, n0 + tn) + d
                    ok = (c >= 0) & (c < sp.ncols)
                    part, pa = np.zeros((tm, tn), LD), np.zeros((tm, tn), LD)
                    part[:, ok] = S[:, c[ok]]; pa[:, ok] = Sa[:, c[ok]]
                    ref += LD(coef) * part; absref += LD(abs(coef)) * pa; N += int(sp.cnt[row0 + m0:row0 + m0 + tm].max()) + 1
        return segs, ref, absref, N

    def shape():
        tm, tn = int(rng.choice(EXTS)), int(rng.choice(EXTS))
        return int(rng.integers(0, CELL - tm + 1)), int(rng.integers(0, CELL - tn + 1)), tm, tn

    for j in range(150):
        m0, n0, tm, tn = shape()
        segs, ref, absref, N = chain(m0, n0, tm, tn, 1 + j % 12)
        where = ("O", "Y", "W")[j % 3]
        mode = int(j % 5 == 4)
        init = rng.standard_normal((tm, tn)) if mode else None
        plan.item(segs, m0, n0, tm, tn, ref, absref, N, where=where, mode=mode, init=init)
    for j in range(24):   # partial tiles in w, summed by run_reduce
        m0, n0, tm, tn = shape()
        nparts = 1 + j % 5
        src = plan.W.tile(nparts * tm, tn, tn)
        tot, tabs, tN = np.zeros((tm, tn), LD), np.zeros((tm, tn), LD), 0
        for p in range(nparts):
            segs, ref, absref, N = chain(m0, n0, tm, tn, 1 + (j + p) % 6)
            b = len(plan.segs)
            plan.segs.extend(segs)
            it = np.zeros(1, ITEM)[0]
            it["C"], it["ldc"], it["m0"], it["n0"], it["tm"], it["tn"] = 8 * (src + p * tm * tn), tn, m0, n0, tm, tn
            it["seg_begin"], it["seg_end"], it["c_in_y"] = b, len(plan.segs), 2
            plan.items.append(it)
            plan.expect.append(("W", src + p * tm * tn, tn, ref, absref, N, None))
            tot += ref; tabs += absref; tN += N
        to_y = bool(j & 1)
        dst = (plan.Y if to_y else plan.O).tile(tm, tn, tn + 2)
        r = np.zeros(1, RED)[0]
        r["dst"], r["ldc"], r["src_off"], r["tm"], r["tn"], r["nparts"], r["dst_in_y"] = 8 * dst if to_y else dst, tn + 2, 8 * src, tm, tn, nparts, int(to_y)
        plan.red.append(r)
        plan.expect.append(("Y" if to_y else "O", dst, tn + 2, tot, tabs, tN + nparts, None))
    return plan


@pytest.mark.parametrize("seed", [0, 1])
def test_chain_mixed_segments_outputs_and_reduce(dc, seed):
    plan = mixed_plan(seed)
    a1 = plan.run(dc)
    plan.check(a1)
    a2 = plan.run(dc)
    for k in "OYW":
        assert (bits(a1[k]) == bits(a2[k])).all(), "two runs of one launch differ"
    # the same launch on the two-stage ring: filler items (copies of the stored plain-output items) up to 1800
    by_off = {e[1]: e for e in plan.expect if e[0] == "O"}
    plain = [it for it in plan.items if it["c_in_y"] == 0 and it["mode"] == 0]
    items = list(plan.items)
    extra, k = [], 0
    while len(items) < DEEP_BELOW + 1:
        it = plain[k % len(plain)].copy()
        _, _, ldc, ref, absref, N, _ = by_off[int(it["C"])]
        it["C"] = plan.O.tile(int(it["tm"]), int(it["tn"]), ldc)
        items.append(it)
        extra.append(("O", int(it["C"]), ldc, ref, absref, N, None))
        k += 1
    a3 = plan.run(dc, items)
    plan.check(a3, plan.expect + extra)
    for key in "YW":
        g = a1["g"]
        assert (bits(a1[key][g:-g]) == bits(a3[key][g:g + a1[key].size - 2 * g])).all(), "the ring depth changed the arithmetic (%s)" % key
    g = a1["g"]
    n1 = a1["O"].size - 2 * g
    assert (bits(a1["O"][g:g + n1 - 1]) == bits(a3["O"][g:g + n1 - 1])).all(), "the ring depth changed the arithmetic (O)"


def test_chain_refuses_plans_past_their_buffers(dc):
    """the shim's own plan validation (both flavours): a GEMM that reads past its operand pool, a tile past its output"""
    plan = ChainPlan()
    A = plan.D.put(np.ones(16))
    s = seg_record(A=A, B=A, lda_m=4, lda_k=1, ldb_n=4, ldb_k=1, coef=1.0, K=4, type=SEG_GEMM)
    plan.item([s], 0, 0, 4, 4, np.zeros((4, 4), LD), np.zeros((4, 4), LD), 5)
    a = plan.arrays()
    a["segs"] = np.array(plan.segs, SEG)
    args = lambda: (a["items"], 1, a["segs"], 1, a["red"], 0, a["g"], a["D"], a["D"].size, a["I"], a["I"].size, a["X"], a["X"].size,
                    a["Y"], a["Y"].size, a["W"], a["W"].size, a["O"], a["O"].size)
    dc.ok("dc_chain", *args())
    a["segs"]["K"] = a["D"].size - 2 * a["g"] - 11         # row 3 of A then reaches the first element past the pool
    assert "outside" in dc.refused("dc_chain", *args())
    a["segs"]["K"] = 4
    a["items"]["C"] = a["O"].size - 2 * a["g"] - 15
    assert "outside" in dc.refused("dc_chain", *args())


def test_emulation_refuses_stager_offsets_past_32_bits():
    """host emulation: a GEMM whose staged element offsets need more than 32 bits is refused (chain_kernel's Stager keeps
    them in int); the nearest legal plan passes"""
    lib = C.CDLL(lib_path("host"))
    msg = C.create_string_buffer(512)
    it = np.zeros(1, ITEM); it["tm"], it["tn"], it["seg_end"] = 64, 64, 1
    sg = np.zeros(1, SEG); sg["type"], sg["K"], sg["coef"] = SEG_GEMM, 16, 1.0
    lim = 2 ** 31 - 1
    for field_row, field_k, ext in (("lda_m", "lda_k", "tm"), ("ldb_n", "ldb_k", "tn")):
        for ld_k, ok in ((lim // 15, True), (lim // 15 + 1, False)):
            s = sg.copy(); s["lda_m"] = s["ldb_n"] = 1; s["lda_k"] = s["ldb_k"] = 1
            s[field_row], s[field_k] = 0, ld_k
            rc = lib.plancheck_check_chain(C.c_void_p(it.ctypes.data), 1, C.c_void_p(s.ctypes.data), msg, 512)
            assert (rc == 0) == ok, (field_k, ld_k, msg.value)
        s = sg.copy(); s["lda_m"] = s["ldb_n"] = 1; s["lda_k"] = s["ldb_k"] = 1
        s[field_row] = (lim - 15) // 63 + 1
        rc = lib.plancheck_check_chain(C.c_void_p(it.ctypes.data), 1, C.c_void_p(s.ctypes.data), msg, 512)
        assert rc != 0 and b"32-bit" in msg.value
    s = sg.copy(); s["K"] = 0; s["lda_m"] = 2 ** 40
    assert lib.plancheck_check_chain(C.c_void_p(it.ctypes.data), 1, C.c_void_p(s.ctypes.data), msg, 512) == 0   # K = 0 stages nothing


# ---------------------------------------------------------------------------------------------------------------------
#  gram
# ---------------------------------------------------------------------------------------------------------------------
def gram_call(dc, P, ldp, np_, n, shift=0):
    g = guard_for(ldp)
    Pf = wrap(P, g)
    Gf = sentinel(np_ * np_, g)
    dc.ok("dc_gram", Pf, Pf.size, ldp, np_, n, shift, Gf, Gf.size, g)
    assert_guards(Gf, g, "G")
    return Gf[g:-g].reshape(np_, np_)


def panel(rng, np_, n, ldp, dyadic):
    """np_ columns of ldp doubles, rows [n, ldp) NaN; dyadic: entries k·2^-12, |k| <= 2^12, so every product and every
    partial sum of a Gram entry (n < 2^28) is exact in float64"""
    P = np.full((np_, ldp), np.nan)
    P[:, :n] = rng.integers(-4096, 4097, (np_, n)) * 2.0 ** -12 if dyadic else rng.standard_normal((np_, n))
    return P.ravel()


GRAM_N = [1, 2, 63, 64, 65, 8191, 8192, 8193, 3 * 8192 + 5]


@pytest.mark.parametrize("np_", [1, 2, 31, 32, 33, 64, 65, 97])
def test_gram_tiles_and_slabs(dc, np_):
    """every 32-column tile edge against every 8192-row slab edge; exact (dyadic) data: G must equal PᵀP exactly, be
    exactly symmetric and give the same bits on a second call"""
    rng = rng_for("gram", np_)
    for n in GRAM_N:
        ldp = n + 2 + (n & 1)       # even, > n
        P = panel(rng, np_, n, ldp, True)
        G = gram_call(dc, P, ldp, np_, n)
        Pm = P.reshape(np_, ldp)[:, :n]
        assert (G == Pm @ Pm.T).all(), (np_, n)
        assert (bits(G) == bits(G.T)).all()
        assert (bits(G) == bits(gram_call(dc, P, ldp, np_, n))).all()


def test_gram_random_data_bound(dc):
    rng = rng_for("gram-random")
    for np_, n in ((33, 8193), (65, 3 * 8192 + 5), (97, 65)):
        ldp = (n + 2) & ~1
        P = panel(rng, np_, n, ldp, False)
        G = gram_call(dc, P, ldp, np_, n)
        Pm = P.reshape(np_, ldp)[:, :n].astype(LD)
        assert_bound(G, Pm @ Pm.T, np.abs(Pm) @ np.abs(Pm).T, n, "gram %dx%d" % (np_, n))
        assert (bits(G) == bits(G.T)).all()


def test_gram_refuses_misaligned_columns(dc):
    rng = rng_for("gram-align")
    P = panel(rng, 3, 10, 12, True)
    g = guard_for(12)
    Pf, Gf = wrap(np.concatenate([P, [0.0]]), g), sentinel(9, g)
    assert "16-byte" in dc.refused("dc_gram", Pf, Pf.size, 12, 3, 10, 1, Gf, Gf.size, g)
    P = panel(rng, 3, 10, 11, True)
    Pf = wrap(P, g)
    assert "16-byte" in dc.refused("dc_gram", Pf, Pf.size, 11, 3, 10, 0, Gf, Gf.size, g)


# ---------------------------------------------------------------------------------------------------------------------
#  gs_pass / gs_final / dot / scale_inv_norm / ritz_rotate
# ---------------------------------------------------------------------------------------------------------------------
NVEC = [1, 4, 5, 8, 9, 12, 13, 17, 18, 24, 25, 39]
NS_SMALL = [1, 255, 256, 257]
NS_BIG = [RED_BLOCKS * 256, RED_BLOCKS * 256 + 1, 10 ** 6 + 3]


def basis(rng, nvec, n, ldv):
    V = np.full((nvec, ldv), np.nan)
    V[:, :n] = rng.standard_normal((nvec, n))
    return V


def gs_pass_call(dc, V, ldv, nvec, w, n, coef, want_dots, want_nrm2):
    g = guard_for(ldv)
    Vf, wf = wrap(V.ravel(), g), wrap(w, g)
    cf = wrap(coef, g) if coef is not None else None
    df = sentinel(nvec, g) if want_dots else None
    rf = sentinel(1, g) if want_nrm2 else None
    dc.ok("dc_gs_pass", Vf, Vf.size, ldv, nvec, wf, wf.size, n, cf, 0 if cf is None else cf.size, df, 0 if df is None else df.size,
          rf, 0 if rf is None else rf.size, g)
    assert (np.isnan(wf[:g]).all() and np.isnan(wf[-g:]).all())
    for f in (df, rf):
        if f is not None:
            assert_guards(f, g)
    return wf[g:-g], None if df is None else df[g:-g], None if rf is None else rf[g:-g][0]


def check_gs_pass(dc, rng, nvec, n, coef_on, dots_on, nrm2_on):
    ldv = n + 3
    V = basis(rng, nvec, n, ldv)
    w = rng.standard_normal(n)
    coef = rng.standard_normal(nvec) if coef_on else None
    wo, dots, nrm2 = gs_pass_call(dc, V, ldv, nvec, w, n, coef, dots_on, nrm2_on)
    Vl = V[:, :n].astype(LD)
    if coef_on:
        ref = w.astype(LD) - coef.astype(LD) @ Vl
        assert_bound(wo, ref, np.abs(w).astype(LD) + np.abs(coef).astype(LD) @ np.abs(Vl), nvec + 1, "gs_pass w")
    else:
        assert (bits(wo) == bits(w)).all(), "gs_pass wrote w without coefficients"
    wl = wo.astype(LD)     # the dot products are of the updated w as stored
    if dots_on:
        assert_bound(dots, Vl @ wl, np.abs(Vl) @ np.abs(wl), n, "gs_pass dots (nvec %d, n %d)" % (nvec, n))
    if nrm2_on:
        assert_bound(nrm2, wl @ wl, wl @ wl, n, "gs_pass nrm2")
    return V, w, coef, wo, dots, nrm2


def test_gs_pass_template_and_block_edges(dc):
    rng = rng_for("gs_pass")
    for nvec in NVEC:
        for n in NS_SMALL + NS_BIG[1:2]:
            check_gs_pass(dc, rng, nvec, n, True, True, True)
    for nvec, n in ((1, NS_BIG[0]), (39, NS_BIG[0]), (4, NS_BIG[2]), (39, NS_BIG[2])):
        check_gs_pass(dc, rng, nvec, n, True, True, True)


def test_gs_pass_null_outputs_and_back_to_back_calls(dc):
    """every combination of coef / dots / nrm2 being null; calls that change n and nvec back to back (a ticket left
    non-zero would leave the next call's outputs unwritten), and two identical calls give the same bits"""
    rng = rng_for("gs_pass-null")
    for n in (257, RED_BLOCKS * 256 + 1):
        for nvec in (5, 24):
            for mask in range(8):
                check_gs_pass(dc, rng, nvec, n, bool(mask & 1), bool(mask & 2), bool(mask & 4))
    V = basis(rng, 18, 70001, 70004)
    w = rng.standard_normal(70001)
    coef = rng.standard_normal(18)
    r1 = gs_pass_call(dc, V, 70004, 18, w, 70001, coef, True, True)
    check_gs_pass(dc, rng, 3, 1, True, True, True)
    r2 = gs_pass_call(dc, V, 70004, 18, w, 70001, coef, True, True)
    for x, y in zip(r1, r2):
        assert (bits(np.atleast_1d(x)) == bits(np.atleast_1d(y))).all()


def test_dot_and_scale_inv_norm(dc):
    rng = rng_for("dot")
    for n in NS_SMALL + NS_BIG:
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        g = guard_for()
        xf, yf, of = wrap(x, g), wrap(y, g), sentinel(1, g)
        dc.ok("dc_dot", xf, xf.size, yf, yf.size, n, of, of.size, g)
        assert_guards(of, g)
        assert_bound(of[g], x.astype(LD) @ y.astype(LD), np.abs(x).astype(LD) @ np.abs(y).astype(LD), n, "dot n=%d" % n)
        nrm2 = float(rng.uniform(0.5, 4.0))
        nf, vf = wrap(np.array([nrm2]), g), sentinel(n, g)
        dc.ok("dc_scale_inv_norm", xf, xf.size, nf, nf.size, vf, vf.size, n, g)
        assert_guards(vf, g)
        ref = x.astype(LD) / np.sqrt(LD(nrm2))
        assert_bound(vf[g:-g], ref, np.abs(ref), 2, "scale_inv_norm")   # a square root, a division and a product


def gs_final_call(dc, V, ldv, nvec, w, n, coef, nin):
    g = guard_for(ldv)
    Vf, wf, cf, nf = wrap(V.ravel(), g), wrap(w, g), wrap(coef, g), wrap(np.array([nin]), g)
    of, vf = sentinel(1, g), sentinel(n, g)
    dc.ok("dc_gs_final", Vf, Vf.size, ldv, nvec, wf, wf.size, n, cf, cf.size, nf, nf.size, of, of.size, vf, vf.size, g)
    assert_guards(of, g); assert_guards(vf, g)
    return of[g], vf[g:-g]


@pytest.mark.parametrize("n", NS_SMALL + NS_BIG)
def test_gs_final_paths(dc, n):
    """the corrected path, the skip path with V all NaN (it must not read V) and b2 <= 0 (vout = 0), for every template
    instance up to MAX_BASIS + 1 vectors"""
    rng = rng_for("gs_final", n)
    nvecs = NVEC + [40] if n < 10 ** 5 else [1, 12, 13, 24, 25, 40] if n < 10 ** 6 else [1, 40]
    for nvec in nvecs:
        ldv = n + 1
        V = basis(rng, nvec, n, ldv)
        w = rng.standard_normal(n)
        coef = 1e-3 * rng.standard_normal(nvec)
        nin = float(w @ w) + 1.0
        b2, v = gs_final_call(dc, V, ldv, nvec, w, n, coef, nin)
        Vl, cl = V[:, :n].astype(LD), coef.astype(LD)
        b2_ref = LD(nin) - cl @ cl
        assert_bound(b2, b2_ref, LD(nin) + cl @ cl, nvec, "gs_final b2")
        num = w.astype(LD) - cl @ Vl
        inv = 1 / np.sqrt(b2_ref)
        assert_bound(v, num * inv, (np.abs(w).astype(LD) + np.abs(cl) @ np.abs(Vl)) * inv, nvec + 3, "gs_final vout (nvec %d)" % nvec)
        # skip path: the correction is below GS_REFINE_REL of the norm; V is never read
        Vn = np.full_like(V, np.nan)
        tiny = np.full(nvec, 1e-14 / np.sqrt(nvec)) * np.sqrt(nin)
        b2s, vs = gs_final_call(dc, Vn, ldv, nvec, w, n, tiny, nin)
        assert b2s == nin
        assert_bound(vs, w.astype(LD) / np.sqrt(LD(nin)), np.abs(w).astype(LD) / np.sqrt(LD(nin)), 2, "gs_final skip path")
        # b2 <= 0: vout is zero
        big = np.full(nvec, np.sqrt(2 * nin / nvec))
        b2z, vz = gs_final_call(dc, V, ldv, nvec, w, n, big, nin)
        assert b2z == 0.0 and (vz == 0.0).all()


@pytest.mark.parametrize("ncv", [1, 4, 5, 8, 9, 12, 13, 17, 18, 24, 25, 39, 40])
def test_ritz_rotate_in_place(dc, ncv):
    rng = rng_for("ritz", ncv)
    for n in (1, 257, RED_BLOCKS * 256 + 1):
        ldv = n + 2
        g = guard_for(ldv)
        if n > 257 and ncv not in (1, 17, 18, 40):
            continue
        for kk in range(1, ncv + 1) if n <= 257 else (ncv,):
            V = basis(rng, ncv, n, ldv)
            S = rng.standard_normal((ncv, kk))
            Vf, Sf = wrap(V.ravel(), g), wrap(S.ravel(), g)
            before = Vf.copy()
            dc.ok("dc_ritz_rotate", Vf, Vf.size, ldv, n, ncv, Sf, Sf.size, kk, g)
            out = Vf[g:-g].reshape(ncv, ldv)
            Vl = V[:, :n].astype(LD)
            assert_bound(out[:kk, :n], S.T.astype(LD) @ Vl, np.abs(S.T).astype(LD) @ np.abs(Vl), ncv, "ritz_rotate ncv %d kk %d" % (ncv, kk))
            mask = np.ones(Vf.size, bool)
            mask[g:-g] = np.ones((ncv, ldv), bool).ravel()
            m2 = np.zeros((ncv, ldv), bool); m2[:kk, :n] = True
            mask[g:-g] &= ~m2.ravel()
            assert_unchanged(Vf, before, mask, "ritz_rotate: V past kk, padding or guards")


def test_basis_limits_are_refused(dc):
    g = guard_for()
    n = 8
    V, w, c = wrap(np.zeros(41 * n), g), wrap(np.zeros(n), g), wrap(np.zeros(41), g)
    r, o = sentinel(41, g), sentinel(n, g)
    nin = wrap(np.ones(1), g)
    assert "gs_pass" in dc.refused("dc_gs_pass", V, V.size, n, MAX_BASIS + 1, w, w.size, n, c, c.size, r, r.size, None, 0, g)
    assert "gs_final" in dc.refused("dc_gs_final", V, V.size, n, MAX_BASIS + 2, w, w.size, n, c, c.size, nin, nin.size, r, r.size, o, o.size, g)
    assert "ritz_rotate" in dc.refused("dc_ritz_rotate", V, V.size, n, n, MAX_BASIS + 2, c, c.size, 1, g)
    # run_spmm: one 1×1 tile without terms, staged for max_nR; the guard covers SP_ROWS·max_nR as dc_spmm requires
    for max_nr, ok in ((SP_MAX_NR + 1, False), (SP_MAX_NR, True)):
        gs = guard_for(SP_ROWS * max_nr)
        tile = np.zeros(1, SP_TILE)
        tile["nR"], tile["nrows"] = 1, 1
        X, Y, I, Vv = wrap(np.zeros(1), gs), sentinel(1, gs), wrap(np.zeros(1, np.int32), gs), wrap(np.zeros(1), gs)
        args = ("dc_spmm", tile, 1, np.zeros(1, SP_ASLOT), 0, np.zeros(1, SP_SSLOT), 0, np.zeros(1, SP_BSLOT), 0, gs, X, X.size, Y, Y.size, I, I.size,
                Vv, Vv.size, max_nr)
        if ok:
            dc.ok(*args)
            assert Y[gs] == 0.0
        else:
            assert "run_spmm" in dc.refused(*args)


# ---------------------------------------------------------------------------------------------------------------------
#  lanczos_batch
# ---------------------------------------------------------------------------------------------------------------------
class BlockH:
    """a symmetric block-diagonal H of dense 4×4 blocks (the last one cut at n), applied in longdouble"""

    def __init__(self, rng, n):
        self.n = n
        nb = (n + 3) // 4
        Hb = rng.standard_normal((nb, 4, 4))
        self.Hb = ((Hb + Hb.transpose(0, 2, 1)) / 2).astype(LD)

    def __call__(self, x):
        xp = np.zeros(self.Hb.shape[0] * 4, LD)
        xp[:self.n] = x
        return np.einsum("kij,kj->ki", self.Hb, xp.reshape(-1, 4)).ravel()[:self.n]


class Lanczos:
    """the device state of one batch: three slots of nb columns (ld > n, NaN padding), per-column scalars"""

    def __init__(self, dc, n, ld, nsteps, starts, zero2):
        self.dc, self.n, self.ld, self.nsteps, self.nb = dc, n, ld, nsteps, len(starts)
        self.g = guard_for(ld)
        nb = self.nb
        self.state = dict(alpha=np.zeros(nb * nsteps), beta=np.zeros(nb * nsteps), norm2=np.zeros(nb), ndone=np.zeros(nb, np.int64),
                          a=np.zeros(nb), scale=np.zeros(nb), zero2=np.asarray(zero2, np.float64), done=np.zeros(nb, np.int32),
                          tickets=np.zeros(nb, np.uint32))
        self.full = {k: wrap(v, self.g) for k, v in self.state.items()}
        self.slots = [self.cols(None), self.cols(None), self.cols(starts)]   # prev, cur, y

    def cols(self, vals):
        a = np.full((self.nb, self.ld), np.nan)
        a[:, :self.n] = 0.0 if vals is None else np.asarray(vals)
        return wrap(a.ravel(), self.g)

    def col(self, slot, c):
        return self.slots[slot][self.g:-self.g].reshape(self.nb, self.ld)[c, :self.n]

    def set_col(self, slot, c, v):
        self.slots[slot][self.g:-self.g].reshape(self.nb, self.ld)[c, :self.n] = v

    def get(self, k):
        return self.full[k][self.g:-self.g]

    def run(self, pass_, t):
        f, g = self.full, self.g
        pads = [s.copy() for s in self.slots]
        self.dc.ok("dc_lanczos", pass_, t, self.nb, self.nsteps, self.n, self.ld, f["alpha"], f["beta"], f["norm2"], f["ndone"], f["a"], f["scale"],
                   f["zero2"], f["done"], f["tickets"], f["norm2"].size, self.slots[0], self.slots[1], self.slots[2], self.slots[0].size, g)
        assert (self.get("tickets") == 0).all(), "tickets left non-zero after pass %d" % pass_
        for s, b in zip(self.slots, pads):   # padding rows and guards untouched
            m = np.ones(s.size, bool)
            inner = np.zeros((self.nb, self.ld), bool); inner[:, :self.n] = True
            m[g:-g] &= ~inner.ravel()
            assert_unchanged(s, b, m, "lanczos columns' padding or guards")

    def rotate(self):
        self.slots = [self.slots[1], self.slots[2], self.slots[0]]


def drive_lanczos(dc, H, n, ld, nsteps, starts, zero2):
    """the caller's side of dev.h's contract, every pass checked against longdouble from its own inputs"""
    L = Lanczos(dc, n, ld, nsteps, starts, zero2)
    nb = len(starts)
    y0 = [L.col(2, c).astype(LD) for c in range(nb)]
    L.run(0, 0)
    done = L.get("done").copy()
    for c in range(nb):
        b2 = y0[c] @ y0[c]
        if done[c]:
            assert L.get("norm2")[c] == 0.0 and b2 <= LD(zero2[c]) * (1 + 4 * LD(U) * n)
        else:
            assert_bound(L.get("norm2")[c], b2, b2, n, "lanczos pass 0")
            assert_bound(L.get("scale")[c], np.sqrt(b2), np.sqrt(b2), n, "lanczos scale")
    L.rotate()   # (prev, cur, y) <- (cur, y, prev): cur = u_0
    for t in range(nsteps):
        act = [c for c in range(nb) if not L.get("done")[c]]
        for c in act:   # y = H·cur
            L.set_col(2, c, H(L.col(1, c).astype(LD)).astype(np.float64))
        u_in = {c: L.col(1, c).astype(LD) for c in act}; y_in = {c: L.col(2, c).astype(LD) for c in act}
        p_in = {c: L.col(0, c).astype(LD) for c in act}; sc = {c: LD(L.get("scale")[c]) for c in act}
        L.run(1, t)
        for c in act:
            v, w = L.col(1, c).astype(LD), L.col(2, c).astype(LD)
            assert_bound(v, u_in[c] / sc[c], np.abs(u_in[c] / sc[c]), 1, "lanczos v")
            wref = y_in[c] / sc[c] - (sc[c] * p_in[c] if t > 0 else 0)
            assert_bound(w, wref, np.abs(y_in[c] / sc[c]) + (np.abs(sc[c] * p_in[c]) if t > 0 else 0), 2, "lanczos w")
            assert_bound(L.get("alpha")[c * nsteps + t], v @ w, np.abs(v) @ np.abs(w), n, "lanczos alpha")
        act = [c for c in act if not L.get("done")[c]]
        if not act:
            break
        v_in = {c: L.col(1, c).astype(LD) for c in act}; w_in = {c: L.col(2, c).astype(LD) for c in act}
        a_in = {c: LD(L.get("a")[c]) for c in act}
        L.run(2, t)
        for c in act:
            y = L.col(2, c).astype(LD)
            assert_bound(y, w_in[c] - a_in[c] * v_in[c], np.abs(w_in[c]) + np.abs(a_in[c] * v_in[c]), 1, "lanczos y")
            if not L.get("done")[c]:
                assert_bound(L.get("beta")[c * nsteps + t + 1], np.sqrt(y @ y), np.sqrt(y @ y), n, "lanczos beta")
        L.rotate()
    return L


def lanczos_reference(H, start, nsteps, zero2):
    """the dev.h recurrence in longdouble on the exact H: norm2, alpha, beta, ndone"""
    y = np.asarray(start, LD)
    b2 = y @ y
    alpha, beta = np.zeros(nsteps, LD), np.zeros(nsteps, LD)
    if b2 <= zero2:
        return LD(0), alpha, beta, 0
    c, prev, u = np.sqrt(b2), np.zeros_like(y), y
    for t in range(nsteps):
        v = u / c
        w = H(v) - (c * prev if t > 0 else 0)
        alpha[t] = v @ w
        if t == nsteps - 1:
            return b2, alpha, beta, nsteps
        w = w - alpha[t] * v
        b = np.sqrt(w @ w)
        if b <= LD(1e-10) * np.sqrt(alpha[t] ** 2 + (c ** 2 if t > 0 else 0)):
            return b2, alpha, beta, t + 1
        beta[t + 1] = b
        prev, u, c = v, w, b
    return b2, alpha, beta, nsteps


@pytest.mark.parametrize("n", [1, 1023, 1024, 1025, RED_BLOCKS * 1024 + 3])
def test_lanczos_batch_passes(dc, n):
    """columns: one below zero2 (done with 0 steps), one inside an invariant subspace (the first 4×4 block: done with at
    most 4 steps), generic ones that finish at nsteps; every pass against longdouble from its inputs, the whole
    recurrence against a longdouble one, and one column alone gives the same bits as inside the batch"""
    rng = rng_for("lanczos", n)
    H = BlockH(rng, n)
    nsteps = 6 if n < 10 ** 5 else 4
    ld = n + 5
    starts = [1e-9 * rng.standard_normal(n)]
    inv = np.zeros(n); inv[:min(4, n)] = rng.standard_normal(min(4, n)); starts.append(inv)
    starts += [rng.standard_normal(n) for _ in range(3)]
    zero2 = [1e-12 * n, 0.0, 0.0, 0.0, 1e-300]
    L = drive_lanczos(dc, H, n, ld, nsteps, starts, zero2)
    alpha = L.get("alpha").reshape(-1, nsteps); beta = L.get("beta").reshape(-1, nsteps)
    for c, s in enumerate(starts):
        nrm2, ra, rb, nd = lanczos_reference(H, s, nsteps, zero2[c])
        assert L.get("ndone")[c] == nd, (c, L.get("ndone")[c], nd)
        assert abs(L.get("norm2")[c] - nrm2) <= 1e-13 * nrm2
        scale = float(np.abs(ra).max() + np.abs(rb).max()) + 1e-300
        assert np.abs(alpha[c, :nd] - ra[:nd]).max(initial=0) <= 1e-11 * scale
        assert np.abs(beta[c, :nd] - rb[:nd]).max(initial=0) <= 1e-11 * scale
    assert L.get("ndone")[0] == 0 and 1 <= L.get("ndone")[1] <= 4
    assert (L.get("ndone")[2:] == (nsteps if n > 4 else 1)).all()
    alone = drive_lanczos(dc, H, n, ld, nsteps, starts[3:4], zero2[3:4])
    assert (bits(alone.get("alpha")) == bits(alpha[3])).all() and (bits(alone.get("beta")) == bits(beta[3])).all()


def test_lanczos_emulation_refuses_short_ld():
    dc = Backend("host", lib_path("host"))
    L = Lanczos(dc, 16, 16, 2, [np.ones(16)] * 2, [0.0, 0.0])
    L.ld = 15
    assert "ld below n" in dc.refused("dc_lanczos", 0, 0, 2, 2, 16, 15, *[L.full[k] for k in ("alpha", "beta", "norm2", "ndone", "a", "scale", "zero2", "done", "tickets")],
                                      L.full["norm2"].size, L.slots[0], L.slots[1], L.slots[2], L.slots[0].size, L.g)


# ---------------------------------------------------------------------------------------------------------------------
#  fill_random, filter_small, axpby_out, gather_rows_reversed
# ---------------------------------------------------------------------------------------------------------------------
def splitmix_fill(n, seed, first):
    with np.errstate(over="ignore"):
        gamma = np.uint64(0x9E3779B97F4A7C15)
        z = np.uint64(seed) + (np.uint64(first) + np.arange(n, dtype=np.uint64)) * gamma
        z = z + gamma
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) / 9007199254740992.0 - 0.5


def fill(dc, n, seed, first):
    g = guard_for()
    xf = sentinel(n, g)
    dc.ok("dc_fill_random", xf, xf.size, n, ("u64", seed), first, g)
    assert_guards(xf, g)
    return xf[g:-g]


def test_fill_random_is_splitmix64_of_the_global_index(dc):
    seed = 0xD1B54A32D192ED03
    for n in (1, 255, 256, 257, RED_BLOCKS * 256, RED_BLOCKS * 256 + 1, 10 ** 6 + 3):
        assert (bits(fill(dc, n, seed, 0)) == bits(splitmix_fill(n, seed, 0))).all(), n
    whole = fill(dc, 400000, 7, 0)
    for first, n in ((0, 1), (1, 255), (12345, 151553), (399999, 1), (250000, 150000)):
        assert (bits(fill(dc, n, 7, first)) == bits(whole[first:first + n])).all(), (first, n)


def test_filter_small_axpby_gather(dc):
    rng = rng_for("stream")
    g = guard_for()
    for n in (1, RED_BLOCKS * 256 - 1, RED_BLOCKS * 256, RED_BLOCKS * 256 + 1):
        x = rng.standard_normal(n) * 10.0 ** rng.integers(-20, 2, n)
        xf = wrap(x, g, "sent")
        dc.ok("dc_filter_small", xf, xf.size, n, 1e-8, g)
        assert_guards(xf, g)
        assert (bits(xf[g:-g]) == bits(np.where(np.abs(x) < 1e-8, 0.0, x))).all()
        a, b = rng.standard_normal(n), rng.standard_normal(n)
        af, bf, of = wrap(a, g), wrap(b, g), sentinel(n, g)
        dc.ok("dc_axpby_out", None, 0, bf, bf.size, -0.7, of, of.size, n, g)
        assert_guards(of, g)
        assert (bits(of[g:-g]) == bits(0.0 + -0.7 * b)).all()
        dc.ok("dc_axpby_out", af, af.size, bf, bf.size, -0.7, of, of.size, n, g)
        assert_guards(of, g)
        assert_bound(of[g:-g], a.astype(LD) + LD(-0.7) * b.astype(LD), np.abs(a).astype(LD) + LD(0.7) * np.abs(b).astype(LD), 1, "axpby_out")
    for n, m in ((1, 1), (24, 7), (769, 200), (769, 769)):   # m·n around the 592-block edge
        src = rng.standard_normal(n * n)
        gg = guard_for(n)
        sf, df = wrap(src, gg), sentinel(m * n, gg)
        dc.ok("dc_gather_rows_reversed", sf, sf.size, n, m, df, df.size, gg)
        assert_guards(df, gg)
        assert (bits(df[gg:-gg]) == bits(src.reshape(n, n)[::-1][:m].ravel())).all()
