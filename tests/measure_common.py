"""Helpers shared by the measurement tests (correlation matrix, dimer matrix, spectral function, dynamical correlations) and
by their probes under tools/: the lattices, the library and driver fixtures, uploaded and exact blocks, exact diagonalisation
and the per-correlator reference path.  A test file imports the fixtures P, ctx and exe by name."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import driver_common as dc
import libswitch
import parity_common as pc

ROOT = dc.ROOT
PLANCHECK = os.path.join(ROOT, "tests", "plancheck", "libdmrgx_plancheck.so")
EXE = {"plancheck": os.path.join(ROOT, "tests", "plancheck", "DMRG-SquareLattice.plancheck.x"),
       "cuda": os.path.join(ROOT, "dmrg.x_b200", "DMRG-SquareLattice.x")}
SM, SZ, SP = -1, 0, 1
J1J2_CYL = dict(Lx=4, Ly=4, J1=0.5, Jz1=1.0, J2=0.25, Jz2=0.5, bcx=0, bcy=1)
HEIS_CHAIN12 = dict(Lx=12, Ly=1, J1=0.5, Jz1=1.0, J2=0.0, Jz2=0.0, bcx=0, bcy=0)

# driver runs on the 4x4 J1-J2 cylinder, and the -mwarmup / -msweeps of each library flavour
DRIVER_RUN = (["-Lx", 4, "-Ly", 4, "-J1", 0.5, "-Jz1", 1, "-J2", 0.25, "-Jz2", 0.5], J1J2_CYL)
DRIVER_M = {"plancheck": (16, [16]), "cuda": (256, [256])}


@pytest.fixture(scope="module", params=["plancheck", pytest.param("cuda", marks=pytest.mark.gpu)])
def P(request):
    import dmrgx_loader
    P = dmrgx_loader.load_package()
    if request.param == "plancheck":
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "dmrg.x_b200", "csrc"), "plancheck"])
        libswitch.use_library(P, PLANCHECK)
    else:
        libswitch.use_library(P, None)
    P.kind = request.param
    yield P
    libswitch.use_library(P, None)


@pytest.fixture()
def ctx(P):
    c = P.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def exe(P):
    if P.kind == "plancheck":
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "dmrg.x_b200", "driver"), "plancheck"])
    assert os.path.exists(EXE[P.kind]), "build it with __graft_entry__.build()"
    return EXE[P.kind]


def ngpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


# ---- blocks and states ---------------------------------------------------------------------------------------------------

def ham_terms(P, ham, nsites):
    return P.HamiltonianTerms(ham["Lx"], ham["Ly"], ham["J1"], ham["Jz1"], ham["J2"], ham["Jz2"], nsites, ham["bcx"], ham["bcy"])


def oracle_blocks(orc, P, ctx, nsites_L, nsites_R, spin_twice=1):
    """oracle warm-up blocks of the 4x4 J1-J2 cylinder, enlarged by one site, uploaded to the product"""
    h = J1J2_CYL
    d = orc.DMRG(h["Lx"], h["Ly"], h["J1"], h["Jz1"], h["J2"], h["Jz2"], spin_twice=spin_twice)
    d.warmup(20)
    enl = lambda k: orc.kron_eye(d.block(k - 2), orc.Block.single_site(spin_twice), pc.lr_terms(orc, h, k))
    pL = pc.upload_block(P, ctx, enl(nsites_L), orc)
    pR = pL if nsites_R == nsites_L else pc.upload_block(P, ctx, enl(nsites_R), orc)
    return pL, pR


def exact_halves(P, ctx, ham):
    """the two un-truncated halves of a lattice (every Sz_i / Sp_i exact) and the terms of the whole lattice"""
    N = ham["Lx"] * ham["Ly"]
    site = P.Block.SingleSite(ctx)
    blk = P.Block.SingleSite(ctx)
    for k in range(2, N // 2 + 1):
        blk = P.KronEye_Explicit(blk, site, ham_terms(P, ham, k))
    return blk, ham_terms(P, ham, N)


def random_psi(ctx, n, seed):
    """a seeded normalised vector: (device vector, host array)"""
    x = np.random.default_rng(seed).standard_normal(n)
    x /= np.linalg.norm(x)
    return ctx.vec(n, x), x


# ---- exact diagonalisation -------------------------------------------------------------------------------------------------

def site_op(N, o, i):
    """single-site spin-1/2 operator on site i of an N-site chain (basis state 0 = up), sparse 2^N × 2^N"""
    import scipy.sparse as sp
    loc = {SZ: np.diag([0.5, -0.5]), SP: np.array([[0.0, 1.0], [0.0, 0.0]]), SM: np.array([[0.0, 0.0], [1.0, 0.0]])}[o]
    return sp.kron(sp.kron(sp.identity(2 ** i), sp.csr_matrix(loc)), sp.identity(2 ** (N - 1 - i)), format="csr")


def exact_diagonalisation(terms, N, k=1):
    """the k lowest energies of the lattice Hamiltonian in the Sz = 0 sector (ascending), its ground state as a full 2^N
    vector, H, the single-site operators {(op, site): matrix} and the number of set bits (down spins) of every basis state"""
    import scipy.sparse.linalg as sla
    ops = {(o, i): site_op(N, o, i) for o in (SZ, SP, SM) for i in range(N)}
    H = sum(a * (ops[(io, i)] @ ops[(jo, j)]) for (a, io, i, jo, j) in terms).tocsr()
    ndown = np.array([bin(b).count("1") for b in range(2 ** N)])   # bit set = down spin, in either convention: Sz = 0 <=> N/2 set
    sec = np.nonzero(ndown == N // 2)[0]
    w, v = sla.eigsh(H[sec][:, sec], k=k, which="SA", tol=1e-14)
    order = np.argsort(w)
    w, v = w[order], v[:, order]
    psi = np.zeros(2 ** N)
    psi[sec] = v[:, 0]
    return w, psi, H, ops, ndown


# ---- the per-correlator path ---------------------------------------------------------------------------------------------

def product_expect(P, kb, dpsi, nL, n, ops):
    """<psi| O_1 O_2 ... |psi> for superblock-site operators [(op, site), ...] through dmrgx_hshell_create_product +
    dmrgx_expect; each block's operators keep their list order (operators of different blocks commute)."""
    lops = [(o, s) for o, s in ops if s < nL]
    rops = [(o, n - 1 - s) for o, s in ops if s >= nL]
    L = P.lib()
    la = np.array([o for o, _ in lops], np.int32); ls = np.array([s for _, s in lops], np.int64)
    ra = np.array([o for o, _ in rops], np.int32); rs = np.array([s for _, s in rops], np.int64)
    h = C.c_void_p()
    assert L.dmrgx_hshell_create_product(kb.h, C.c_longlong(len(lops)), la.ctypes.data_as(C.c_void_p), ls.ctypes.data_as(C.c_void_p),
                                         C.c_longlong(len(rops)), ra.ctypes.data_as(C.c_void_p), rs.ctypes.data_as(C.c_void_p), C.byref(h)) == 0, \
        L.dmrgx_last_error()
    v = C.c_double()
    assert L.dmrgx_expect(h, dpsi.ptr, C.byref(v)) == 0
    L.dmrgx_hshell_destroy(h)
    return v.value


# D_a = Sz_i Sz_j + ½ S+_i S-_j + ½ S-_i S+_j, as (O_i, O_j, coefficient); the transpose of O
DIMER_TERMS = ((SZ, SZ, 1.0), (SP, SM, 0.5), (SM, SP, 0.5))
TRANSPOSE = {SZ: SZ, SP: SM, SM: SP}


def per_correlator_dimer(P, kb, dpsi, nL, n, a, b=None):
    """<psi| D_a |psi>, or <D_a psi, D_b psi> as the 9 products [O_jᵀ, O_iᵀ, O_k, O_l] of the per-correlator path"""
    i, j = a
    if b is None:
        return sum(c * product_expect(P, kb, dpsi, nL, n, [(oi, i), (oj, j)]) for oi, oj, c in DIMER_TERMS)
    k, l_ = b
    return sum(ca * cb * product_expect(P, kb, dpsi, nL, n, [(TRANSPOSE[oj], j), (TRANSPOSE[oi], i), (ok, k), (ol, l_)])
               for oi, oj, ca in DIMER_TERMS for ok, ol, cb in DIMER_TERMS)


def nn_bonds(ham):
    """the distinct nearest-neighbour bonds in NeighborPairs order (1-D snake numbering), with orientation and origin: the site
    from which the +x / +y step leads, for a wrap-around bond the one in the last column / row (a two-leg rung: y = 0)"""
    Lx, Ly = ham["Lx"], ham["Ly"]
    to1d = lambda x, y: x * Ly + y if x % 2 == 0 else (x + 1) * Ly - (y + 1)
    xy = {}
    for x in range(Lx):
        for y in range(Ly):
            xy[to1d(x, y)] = (x, y)
    out = []
    for s in range(Lx * Ly):
        x, y = xy[s]
        nbr = []
        if y < Ly - 1 or ham["bcy"]:
            nbr.append(("y", to1d(x, (y + 1) % Ly)))
        if x < Lx - 1 or ham["bcx"]:
            nbr.append(("x", to1d((x + 1) % Lx, y)))
        for o, t in nbr:
            p = (min(s, t), max(s, t))
            if t == s or p in [b[0] for b in out]:
                continue
            u = {"x": 0, "y": 1}[o]
            a, b = xy[p[0]], xy[p[1]]
            origin = a if a[u] + 1 == b[u] else b if b[u] + 1 == a[u] else max(a, b, key=lambda c: c[u])
            out.append((p, o, origin))
    return out


# ---- the continued-fraction recurrence -----------------------------------------------------------------------------------

def kron_index(kb, nR):
    """full L⊗R index (a·NR + b) of every state of a Kron, in the Kron's order"""
    qn, il, ir, sz, off = kb.data()
    Lq, Ls = kb.left.sectors()
    Rq, Rs = kb.right.sectors()
    Lo, Ro = np.concatenate([[0], np.cumsum(Ls)]), np.concatenate([[0], np.cumsum(Rs)])
    idx = []
    for p in range(len(qn)):
        for a in range(Lo[il[p]], Lo[il[p] + 1]):
            idx.extend(a * nR + np.arange(Ro[ir[p]], Ro[ir[p] + 1]))
    return np.array(idx, np.int64)


def start_vectors(kb, tk, psi, op, coef):
    """phi_v = Σ_s coef[v, s] O_s psi on the target Kron, from the dense block operators embedded with the Kron offsets"""
    L, R = kb.left, kb.right
    nL, nR = L.NumSites(), R.NumSites()
    NL, NR = L.NumStates(), R.NumStates()
    dense = lambda blk, i: pc.dense_op(blk, SP, i).T if op == SM else pc.dense_op(blk, op, i)
    full = np.zeros(NL * NR)
    full[kron_index(kb, NR)] = psi
    X = full.reshape(NL, NR)
    panels = []
    for s in range(nL + nR):
        Y = dense(L, s) @ X if s < nL else X @ dense(R, nL + nR - 1 - s).T
        panels.append(Y.reshape(-1)[kron_index(tk, NR)])
    return np.asarray(coef) @ np.array(panels)


def dense_shell(shell, n):
    return np.array([shell.MatMult_host(e) for e in np.eye(n)]).T


def tridiag(a, b, k):
    return np.diag(a[:k]) + np.diag(b[1:k], 1) + np.diag(b[1:k], -1)
