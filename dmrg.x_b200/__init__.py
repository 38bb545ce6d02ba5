"""dmrgx_b200 — Python plumbing over the C ABI of the B200 superblock path (include/dmrgx.h).

This module is *only* a ctypes binding: device memory, streams and torch.distributed are plumbing, the
product is ``libdmrgx_b200.so`` (hand-written sm_100a kernels behind a C ABI).  The directory is called
``dmrg.x_b200`` (not importable by name); load it with ``load_package()`` from ``dmrgx_loader.py`` at the
repo root, which registers it as ``dmrgx_b200``.

The class and method names mirror the reference: ``Block`` <-> ``Block::SpinBase``
(include/DMRGBlock.hpp:79), ``KronBlocks`` <-> ``KronBlocks_t`` (include/DMRGKron.hpp:117),
``HShell`` <-> the KronSumShell ``Mat`` (src/DMRGKron.cpp:1827-1917).

There is no CPU fallback: without the CUDA library or without a GPU every entry point raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdmrgx_b200.so")

OpSm, OpSz, OpSp, OpEye, OpH = -1, 0, 1, 2, 3

LL = C.c_longlong
_lib = None


class DmrgxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("dmrgx error %d: %s" % (code, msg))
        self.code = code


class EigsOpts(C.Structure):
    _fields_ = [("tol", C.c_double), ("ncv", LL), ("max_it", LL), ("seed", C.c_ulonglong)]


class EigsStats(C.Structure):
    _fields_ = [("nmatvec", LL), ("nrestart", LL), ("converged", LL), ("resid", C.c_double)]


def lib():
    global _lib
    if _lib is None:
        path = LIB_PATH   # the CUDA library next to this file and nothing else (tests/libswitch.py re-points it for CPU-only host-logic tests)
        if not os.path.exists(path):
            raise DmrgxError(100, "%s is missing: build it with __graft_entry__.build() (there is no CPU fallback)" % path)
        L = C.CDLL(path)
        L.dmrgx_last_error.restype = C.c_char_p
        for n in ("dmrgx_ham_terms", "dmrgx_launch_count", "dmrgx_kron_size", "dmrgx_kron_num_states", "dmrgx_kron_map", "dmrgx_kron_offsets_lr"):
            getattr(L, n).restype = LL
        _lib = L
    return _lib


def _chk(code):
    if code:
        raise DmrgxError(code, lib().dmrgx_last_error().decode())


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _l(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _i(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def launch_count():
    return lib().dmrgx_launch_count()


def _terms_arrays(terms):
    return (_d([t[0] for t in terms]), _i([t[1] for t in terms]), _l([t[2] for t in terms]), _i([t[3] for t in terms]),
            _l([t[4] for t in terms]))


def HamiltonianTerms(Lx, Ly, J1=1.0, Jz1=0.0, J2=1.0, Jz2=0.0, nsites=-1, bcx=0, bcy=1, heisenberg=None):
    """Hamiltonians::J1J2XXZModel_SquareLattice::H(nsites) — src/Hamiltonians.cpp:73-122; defaults and the
    -heisenberg override follow include/Hamiltonians.hpp:93-115, 240-265."""
    if heisenberg is not None:
        Jz1, J1, J2, Jz2 = heisenberg, 0.5, 0.0, 0.0
    cap = 16 * max(Lx * Ly, 1) * 3 + 16
    a = np.zeros(cap); iop = np.zeros(cap, np.int32); isite = np.zeros(cap, np.int64); jop = np.zeros(cap, np.int32)
    jsite = np.zeros(cap, np.int64)
    k = lib().dmrgx_ham_terms(LL(Lx), LL(Ly), C.c_double(J1), C.c_double(Jz1), C.c_double(J2), C.c_double(Jz2), int(bcx), int(bcy),
                              LL(nsites), LL(cap), _p(a), _p(iop), _p(isite), _p(jop), _p(jsite))
    assert k <= cap
    return [(float(a[i]), int(iop[i]), int(isite[i]), int(jop[i]), int(jsite[i])) for i in range(k)]


def dist_unique_id():
    """128-byte communicator id (an ncclUniqueId): rank 0 creates it, the launcher broadcasts it (dmrgx_dist_unique_id)."""
    buf = C.create_string_buffer(128)
    _chk(lib().dmrgx_dist_unique_id(buf))
    return buf.raw


class Context:
    """One CUDA device + stream (stands in for the MPI communicator of the reference objects).  With world > 1 this is
    one rank of a multi-GPU job (one process per GPU): objects created on it are sharded by superblock row ranges."""

    def __init__(self, device=0, stream=None, rank=0, world=1, unique_id=None):
        h = C.c_void_p()
        if world > 1:
            assert unique_id is not None and len(unique_id) == 128
            _chk(lib().dmrgx_ctx_create_dist(int(device), C.c_void_p(stream or 0), int(rank), int(world), C.c_char_p(unique_id), C.byref(h)))
        else:
            _chk(lib().dmrgx_ctx_create(int(device), C.c_void_p(stream or 0), C.byref(h)))
        self.h = h
        self.device = device
        self.rank, self.world = rank, world

    def sync(self):
        _chk(lib().dmrgx_ctx_sync(self.h))

    def set_dense_threshold(self, fill):
        _chk(lib().dmrgx_ctx_set_dense_threshold(self.h, C.c_double(fill)))

    def close(self):
        if getattr(self, "h", None):
            lib().dmrgx_ctx_destroy(self.h)
            self.h = None

    # ---- device vectors ----
    def vec(self, n, host=None):
        v = DeviceVector(self, n)
        if host is not None:
            v.set(host)
        return v


class DeviceVector:
    def __init__(self, ctx, n):
        self.ctx, self.n = ctx, int(n)
        p = C.c_void_p()
        _chk(lib().dmrgx_vec_alloc(ctx.h, LL(self.n), C.byref(p)))
        self.ptr = p

    def set(self, host):
        host = _d(host)
        assert host.size == self.n
        _chk(lib().dmrgx_vec_set(self.ctx.h, self.ptr, _p(host), LL(self.n)))

    def get(self):
        out = np.zeros(self.n)
        _chk(lib().dmrgx_vec_get(self.ctx.h, _p(out), self.ptr, LL(self.n)))
        return out

    def __del__(self):
        if getattr(self, "ptr", None) and getattr(self.ctx, "h", None):
            lib().dmrgx_vec_free(self.ctx.h, self.ptr)
            self.ptr = None


class Block:
    """Block::SpinBase on the device (include/DMRGBlock.hpp:79-434)."""

    def __init__(self, ctx, handle):
        self.ctx = ctx
        self.h = handle

    def __del__(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            lib().dmrgx_block_destroy(self.h)
            self.h = None

    @staticmethod
    def Initialize(ctx, nsites, qn_list, qn_size):
        """Initialize(comm, nsites, qn_list, qn_size) — include/DMRGBlock.hpp:243-250"""
        qn = _d(qn_list); sz = _l(qn_size)
        h = C.c_void_p()
        _chk(lib().dmrgx_block_create(ctx.h, LL(nsites), LL(len(qn)), _p(qn), _p(sz), C.byref(h)))
        return Block(ctx, h)

    @staticmethod
    def SingleSite(ctx, spin_twice=1):
        """Initialize(comm, 1, PETSC_DEFAULT) — src/DMRGBlock.cpp:123-137"""
        h = C.c_void_p()
        _chk(lib().dmrgx_block_single_site(ctx.h, int(spin_twice), C.byref(h)))
        return Block(ctx, h)

    @staticmethod
    def InitializeFromDisk(ctx, block_path):
        """InitializeFromDisk(comm, block_path) — src/DMRGBlock.cpp:214-372: BlockInfo.dat, QuantumNumbers.dat and the PETSc
        binary AIJ files Sz_%09d.mat / Sp_%09d.mat / H_000000000.mat (big-endian classid 1211216, M, N, nz, row lengths,
        columns, values) of a block directory written by the reference or by DMRG-SquareLattice.x -scratch_dir."""
        if not block_path.endswith("/"):
            block_path += "/"
        info = dict(l.split()[:2] for l in open(block_path + "BlockInfo.dat") if l.strip())
        ib = int(info["NumBytesPetscInt"])
        if int(info["NumBytesPetscScalar"]) != 8 or int(info["PetscUseComplex"]) != 0 or ib not in (4, 8):
            raise DmrgxError(1, "incompatible BlockInfo.dat in " + block_path)
        rows = [l.split() for l in open(block_path + "QuantumNumbers.dat") if l.strip()]
        blk = Block.Initialize(ctx, int(info["NumSites"]), [float(q) for _, q in rows], [int(s) for s, _ in rows])
        it = np.dtype(">i4" if ib == 4 else ">i8")

        def load(name, isite):
            raw = open("%s%s_%09d.mat" % (block_path, name, isite), "rb").read()
            hdr = np.frombuffer(raw, it, 4)
            if hdr[0] != 1211216 or hdr[1] != blk.NumStates() or hdr[2] != blk.NumStates():
                raise DmrgxError(62, "not a PETSc binary matrix of this block: %s_%09d.mat" % (name, isite))
            M, nz = int(hdr[1]), int(hdr[3])
            off = 4 * ib
            rowlen = np.frombuffer(raw, it, M, off).astype(np.int64); off += M * ib
            col = np.frombuffer(raw, it, nz, off).astype(np.int64); off += nz * ib
            val = np.frombuffer(raw, ">f8", nz, off).astype(np.float64)
            return np.concatenate([[0], np.cumsum(rowlen)]), col, val
        for i in range(blk.NumSites()):
            blk.set_operator(OpSz, i, *load("Sz", i))
            blk.set_operator(OpSp, i, *load("Sp", i))
        if os.path.exists("%sH_%09d.mat" % (block_path, 0)):
            blk.set_operator(OpH, 0, *load("H", 0))
        _chk(blk.CheckOperatorBlocks())
        return blk

    def set_operator(self, op, isite, rowptr, col, val):
        rowptr = _l(rowptr); col = _l(col); val = _d(val)
        _chk(lib().dmrgx_block_set_operator(self.h, int(op), LL(isite), _p(rowptr), _p(col), _p(val)))

    def get_operator(self, op, isite=0):
        nnz = LL()
        _chk(lib().dmrgx_block_get_operator(self.h, int(op), LL(isite), C.byref(nnz), None, None, None))
        n = self.NumStates()
        rowptr = np.zeros(n + 1, np.int64); col = np.zeros(max(nnz.value, 1), np.int64); val = np.zeros(max(nnz.value, 1))
        _chk(lib().dmrgx_block_get_operator(self.h, int(op), LL(isite), C.byref(nnz), _p(rowptr), _p(col), _p(val)))
        return rowptr, col[:nnz.value], val[:nnz.value]

    def get_operator_dense(self, op, isite=0):
        rowptr, col, val = self.get_operator(op, isite)
        n = self.NumStates()
        D = np.zeros((n, n))
        for r in range(n):
            D[r, col[rowptr[r]:rowptr[r + 1]]] = val[rowptr[r]:rowptr[r + 1]]
        return D

    def _info(self):
        a, b, c = LL(), LL(), LL()
        _chk(lib().dmrgx_block_info(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def NumSites(self):
        return self._info()[0]

    def NumStates(self):
        return self._info()[1]

    def sectors(self):
        """Magnetization.List(), Magnetization.Sizes()"""
        ns = self._info()[2]
        qn = np.zeros(ns); sz = np.zeros(ns, np.int64)
        _chk(lib().dmrgx_block_sectors(self.h, _p(qn), _p(sz)))
        return qn, sz

    def CheckOperatorBlocks(self):
        return lib().dmrgx_block_check(self.h)


def KronEye_Explicit(left, site, terms):
    """KronEye_Explicit(LeftBlock, AddSite, Terms, BlockOut) — src/DMRGKron.cpp:459-615"""
    a, iop, isite, jop, jsite = _terms_arrays(terms)
    h = C.c_void_p()
    _chk(lib().dmrgx_block_enlarge(left.h, site.h, LL(len(terms)), _p(a), _p(iop), _p(isite), _p(jop), _p(jsite), C.byref(h)))
    return Block(left.ctx, h)


class KronBlocks:
    """KronBlocks_t (include/DMRGKron.hpp:117-480)."""

    def __init__(self, left, right, qn_sectors):
        self.left, self.right, self.ctx = left, right, left.ctx
        qn = _d(qn_sectors)
        h = C.c_void_p()
        _chk(lib().dmrgx_kron_create(left.h, right.h, LL(len(qn)), _p(qn), C.byref(h)))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            lib().dmrgx_kron_destroy(self.h)
            self.h = None

    def size(self):
        return lib().dmrgx_kron_size(self.h)

    def NumStates(self):
        return lib().dmrgx_kron_num_states(self.h)

    def data(self):
        n = self.size()
        qn = np.zeros(n); il = np.zeros(n, np.int64); ir = np.zeros(n, np.int64); sz = np.zeros(n, np.int64)
        off = np.zeros(n + 1, np.int64)
        _chk(lib().dmrgx_kron_data(self.h, _p(qn), _p(il), _p(ir), _p(sz), _p(off)))
        return qn, il, ir, sz, off

    def Map(self, l, r):
        return lib().dmrgx_kron_map(self.h, LL(l), LL(r))

    def Offsets(self, l, r):
        return lib().dmrgx_kron_offsets_lr(self.h, LL(l), LL(r))

    def KronSumConstruct(self, terms):
        """KronSumConstruct(Terms, H) with the shell matrix — src/DMRGKron.cpp:759-841"""
        return HShell(self, terms=terms)

    def KronConstruct(self, op_left, isite_left, op_right, isite_right):
        """KronConstruct(Mat_L, OpType_L, Mat_R, OpType_R, MatOut) — include/DMRGKron.hpp:309"""
        return HShell(self, single=(op_left, isite_left, op_right, isite_right))

    def CorrelationMatrix(self, psi):
        """EXTENSION (dmrgx_corr_matrix): every two-point spin correlator of psi (a DeviceVector of this superblock) in one
        batched device pass.  Returns a dict of numpy arrays over the superblock sites (site s < nL: left-block site s, else
        right-block site nL+nR-1-s): SzSz, SpSm, SmSp (n×n, entry [i, j] = <psi| O_i O'_j |psi>), Sz (n), and the algorithmic
        flops of the call."""
        n = self.left.NumSites() + self.right.NumSites()
        out = {k: np.zeros((n, n)) for k in ("SzSz", "SpSm", "SmSp")}
        sz = np.zeros(n)
        fl = C.c_double()
        _chk(lib().dmrgx_corr_matrix(self.h, psi.ptr if psi is not None else None, _p(out["SzSz"]), _p(out["SpSm"]), _p(out["SmSp"]), _p(sz),
                                     C.byref(fl)))
        out["Sz"] = sz
        out["flops"] = fl.value
        return out

    def DimerMatrix(self, psi, bonds):
        """EXTENSION (dmrgx_dimer_matrix): every bond–bond correlator of psi over `bonds`, a sequence of (i, j) superblock-site
        pairs, in one batched device pass, with D_a = Sz_i Sz_j + (S+_i S-_j + S-_i S+_j)/2 in the given order.  Returns
        DD (nb×nb, entry [a, b] = <D_a psi, D_b psi>), D (nb, <psi| D_a |psi>) and the algorithmic flops of the call."""
        b = _l(bonds).reshape(-1, 2) if len(bonds) else np.zeros((0, 2), np.int64)
        si, sj = _l(b[:, 0]), _l(b[:, 1])
        nb = len(b)
        dd = np.zeros((nb, nb))
        d = np.zeros(nb)
        fl = C.c_double()
        _chk(lib().dmrgx_dimer_matrix(self.h, psi.ptr if psi is not None else None, LL(nb), _p(si), _p(sj), _p(dd), _p(d), C.byref(fl)))
        return {"DD": dd, "D": d, "flops": fl.value}

    def SpectralLanczos(self, psi, target, op, coef, nsteps, overlaps=False):
        """EXTENSION (dmrgx_spectral_lanczos): continued-fraction coefficients of the start vectors phi_v = Σ_s coef[v, s] O_s psi
        (O = Sz, S+ or S- for op = OpSz, OpSp, OpSm; coef an nvec×n array over the superblock sites) under `target`, an HShell on
        the sector qn + op of the same two blocks.  Returns alpha and beta (nvec×nsteps, beta[:, 0] = 0), norm2 (nvec),
        nsteps_done (nvec) and the algorithmic flops of the call; evaluate G(z) with continued_fraction().
        overlaps=True (dmrgx_spectral_lanczos_overlaps) also returns overlaps (nvec×nsteps×n): <O_s psi, v_t> of every
        Lanczos vector with every site's panel, 0 past nsteps_done; evaluate the cross correlations with
        dynamical_correlation() and time_correlation()."""
        n = self.left.NumSites() + self.right.NumSites()
        c = _d(coef).reshape(-1, n) if np.size(coef) else np.zeros((0, n))
        nvec, nsteps = len(c), int(nsteps)
        alpha = np.zeros((nvec, max(nsteps, 0))); beta = np.zeros((nvec, max(nsteps, 0)))
        norm2 = np.zeros(nvec); done = np.zeros(nvec, np.int64)
        fl = C.c_double()
        args = (self.h, psi.ptr if psi is not None else None, target.h if target is not None else None, int(op), LL(nvec), _p(c), LL(nsteps),
                _p(alpha), _p(beta), _p(norm2), _p(done))
        r = {"alpha": alpha, "beta": beta, "norm2": norm2, "nsteps_done": done}
        if overlaps:
            ov = np.zeros((nvec, max(nsteps, 0), n))
            _chk(lib().dmrgx_spectral_lanczos_overlaps(*args, _p(ov), C.byref(fl)))
            r["overlaps"] = ov
        else:
            _chk(lib().dmrgx_spectral_lanczos(*args, C.byref(fl)))
        r["flops"] = fl.value
        return r


def continued_fraction(alpha, beta, norm2, nsteps_done, z):
    """G(z) = norm2 / (z - α_0 - β_1² / (z - α_1 - … - β_{k-1}² / (z - α_{k-1}))), k = nsteps_done, for one vector (alpha, beta of
    length >= k, scalar norm2 and k) or a batch (nvec×nsteps arrays, nvec norms and counts), at a scalar or a vector of complex z.
    A vector with k = 0 gives 0.  With z = ω + E0 + iη, -Im G / π is the spectral function broadened by a Lorentzian of width η."""
    a, b = np.atleast_2d(np.asarray(alpha, float)), np.atleast_2d(np.asarray(beta, float))
    nrm, k = np.atleast_1d(np.asarray(norm2, float)), np.atleast_1d(np.asarray(nsteps_done, np.int64))
    zz = np.atleast_1d(np.asarray(z, complex))
    G = np.zeros((len(nrm), len(zz)), complex)
    for v in range(len(nrm)):
        g = np.zeros(len(zz), complex)
        for t in range(int(k[v]) - 1, -1, -1):
            g = 1.0 / (zz - a[v, t] - (b[v, t + 1] ** 2 * g if t + 1 < k[v] else 0.0))
        G[v] = nrm[v] * g if k[v] > 0 else 0.0
    if np.ndim(norm2) == 0:
        G = G[0]
    return G if np.ndim(z) else G[..., 0]


def _cross(r, phases):
    """‖phi_v‖ Σ_t ov[v, t, s]·[f(T_v)]_{t,0} with f(θ) = phases(θ) (one row per evaluation point), through one eigh of T_v"""
    ov = np.asarray(r["overlaps"], float)
    nvec, _, n = ov.shape
    out = None
    for v in range(nvec):
        k = int(r["nsteps_done"][v])
        if k == 0:
            f = phases(np.zeros(0))
            res = np.zeros((n, f.shape[0]), f.dtype)
        else:
            a, b = np.asarray(r["alpha"][v], float), np.asarray(r["beta"][v], float)
            th, Y = np.linalg.eigh(np.diag(a[:k]) + np.diag(b[1:k], 1) + np.diag(b[1:k], -1))
            f = phases(th)                                     # (npoints, k)
            res = np.sqrt(r["norm2"][v]) * ((ov[v, :k].T @ Y) * Y[0]) @ f.T
        if out is None:
            out = np.zeros((nvec, n, res.shape[1]), res.dtype)
        out[v] = res
    return out


def dynamical_correlation(r, z):
    """<O_s psi| (z - H)^-1 |phi_v> ≈ ‖phi_v‖ Σ_t ov[v, t, s]·[(z - T_v)^-1]_{t,0} from a SpectralLanczos(..., overlaps=True) result
    r, as an (nvec, n, len(z)) complex array (z a scalar: (nvec, n)).  With site sources (coef rows e_c) and z = ω + E0 + iη,
    -Im / π is the site-resolved S_sc(ω) broadened by a Lorentzian of width η.  A vector with 0 steps gives 0."""
    zz = np.atleast_1d(np.asarray(z, complex))
    G = _cross(r, lambda th: 1.0 / (zz[:, None] - th[None, :]))
    return G if np.ndim(z) else G[..., 0]


def time_correlation(r, times, e0):
    """<O_s psi| e^{-i(H - E0)τ} |phi_v> ≈ ‖phi_v‖ Σ_t ov[v, t, s]·[e^{-i(T_v - E0)τ}]_{t,0} for every τ in times, from a
    SpectralLanczos(..., overlaps=True) result r, as an (nvec, n, len(times)) complex array (a scalar τ: (nvec, n)).  With op Sz
    and site sources this is G_sc(τ) = <S^z_s(τ) S^z_c>.  A vector with 0 steps gives 0."""
    tt = np.atleast_1d(np.asarray(times, float))
    G = _cross(r, lambda th: np.exp(-1j * np.outer(tt, th - e0)))
    return G if np.ndim(times) else G[..., 0]


class HShell:
    """The matrix-free superblock Hamiltonian (MATSHELL with MatMult_KronSumShell)."""

    def __init__(self, kron, terms=None, single=None):
        self.kron, self.ctx = kron, kron.ctx
        h = C.c_void_p()
        if single is not None:
            _chk(lib().dmrgx_hshell_create_single(kron.h, int(single[0]), LL(single[1]), int(single[2]), LL(single[3]), C.byref(h)))
        else:
            a, iop, isite, jop, jsite = _terms_arrays(terms)
            _chk(lib().dmrgx_hshell_create(kron.h, LL(len(terms)), _p(a), _p(iop), _p(isite), _p(jop), _p(jsite), C.byref(h)))
        self.h = h
        self.n = kron.NumStates()

    def __del__(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            lib().dmrgx_hshell_destroy(self.h)
            self.h = None

    def stats(self):
        n, nt, t1, t2 = LL(), LL(), LL(), LL()
        ab, af = C.c_double(), C.c_double()
        _chk(lib().dmrgx_hshell_stats(self.h, C.byref(n), C.byref(nt), C.byref(ab), C.byref(af), C.byref(t1), C.byref(t2)))
        gb, gf, wb = C.c_double(), C.c_double(), C.c_double()
        _chk(lib().dmrgx_hshell_stats_global(self.h, C.byref(gb), C.byref(gf)))
        _chk(lib().dmrgx_hshell_workspace_bytes(self.h, C.byref(wb)))
        return dict(nstates=n.value, nterms=nt.value, alg_bytes=ab.value, alg_flops=af.value, tiles_stage1=t1.value, tiles_stage2=t2.value,
                    alg_bytes_global=gb.value, alg_flops_global=gf.value, workspace_bytes=wb.value)

    def MatMult(self, x, y):
        """MatMult(H, x, y) on device vectors (or raw device pointers as ints)"""
        xp = x.ptr if isinstance(x, DeviceVector) else C.c_void_p(int(x))
        yp = y.ptr if isinstance(y, DeviceVector) else C.c_void_p(int(y))
        _chk(lib().dmrgx_hshell_apply(self.h, xp, yp))

    def row_range(self):
        """(begin, end, cuts): superblock rows this rank owns and the ownership table of all ranks"""
        b, e = LL(), LL()
        cuts = np.zeros(self.ctx.world + 1, np.int64)
        _chk(lib().dmrgx_hshell_row_range(self.h, C.byref(b), C.byref(e), _p(cuts)))
        return b.value, e.value, cuts

    def halo_bytes(self):
        """(bytes of psi this rank receives per sharded apply, what an all-gather would bring)"""
        a, b = C.c_double(), C.c_double()
        _chk(lib().dmrgx_hshell_halo_bytes(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def MatMult_sharded(self, x, y):
        """distributed MatMult: x holds this rank's rows on entry (full-length buffer), receives the sector halo its
        tiles read in place, then this rank's rows of y are computed"""
        _chk(lib().dmrgx_hshell_apply_sharded(self.h, x.ptr, y.ptr))

    def MatMult_stage(self, stage, x, y):
        _chk(lib().dmrgx_hshell_apply_stage(self.h, int(stage), x.ptr, y.ptr))

    def stage_flops(self):
        a, b = C.c_double(), C.c_double()
        _chk(lib().dmrgx_hshell_stage_flops(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def stage_exec_flops(self):
        a, b = C.c_double(), C.c_double()
        _chk(lib().dmrgx_hshell_stage_exec_flops(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def MatMult_host(self, x, y=None):
        """The PETSc-callback shape: host arrays in and out (H2D + kernels + D2H inside).  On a multi-GPU context x and y
        are this rank's local rows (VecGetArray of an MPI Vec)."""
        x = _d(x)
        if y is None:
            b, e, _ = self.row_range()
            y = np.zeros(e - b)
        _chk(lib().dmrgx_hshell_apply_host(self.h, _p(x), _p(y)))
        return y

    def EPSSolve(self, tol=1e-8, ncv=16, max_it=0, seed=20261018, psi=None, initial=None):
        """EPSSolve + EPSGetEigenpair(0) — include/DMRGBlockContainer.hpp:1484-1500.  `initial` (a DeviceVector of the global
        length) is the extension dmrgx_eigs_smallest_from: the reference always starts from a random vector."""
        if psi is None:
            psi = DeviceVector(self.ctx, self.n)
        o = EigsOpts(tol, ncv, max_it, seed)
        s = EigsStats()
        e0 = C.c_double()
        if initial is None:
            _chk(lib().dmrgx_eigs_smallest(self.h, C.byref(o), C.byref(e0), psi.ptr, C.byref(s)))
        else:
            _chk(lib().dmrgx_eigs_smallest_from(self.h, C.byref(o), initial.ptr, C.byref(e0), psi.ptr, C.byref(s)))
        return e0.value, psi, dict(nmatvec=s.nmatvec, nrestart=s.nrestart, converged=bool(s.converged), resid=s.resid)

    def expect(self, psi):
        v = C.c_double()
        _chk(lib().dmrgx_expect(self.h, psi.ptr, C.byref(v)))
        return v.value


class BasisTransformation:
    """BasisTransformation (include/DMRGBlockContainer.hpp:226-257): RotMatT, QN, TruncErr."""

    def __init__(self, ctx, handle):
        self.ctx, self.h = ctx, handle
        m, n, ns, ne = LL(), LL(), LL(), LL()
        te = C.c_double()
        _chk(lib().dmrgx_xform_info(self.h, C.byref(m), C.byref(n), C.byref(ns), C.byref(te), C.byref(ne)))
        self.m, self.nstates, self.nsectors, self.TruncErr, self.nspec = m.value, n.value, ns.value, te.value, ne.value

    def __del__(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            lib().dmrgx_xform_destroy(self.h)
            self.h = None

    def sectors(self):
        qn = np.zeros(self.nsectors); sz = np.zeros(self.nsectors, np.int64)
        _chk(lib().dmrgx_xform_sectors(self.h, _p(qn), _p(sz)))
        return qn, sz

    def spectrum(self):
        ev = np.zeros(self.nspec); bi = np.zeros(self.nspec, np.int64)
        _chk(lib().dmrgx_xform_spectrum(self.h, _p(ev), _p(bi)))
        return ev, bi

    def RotMatT(self):
        out = np.zeros((self.m, self.nstates))
        _chk(lib().dmrgx_xform_rotmat(self.h, _p(out)))
        return out


def GetTruncation(kron, psi, mstates):
    """GetTruncation(KronBlocks, gsv_r, MStates, BT_L, BT_R) — include/DMRGBlockContainer.hpp:1656-1959"""
    l, r = C.c_void_p(), C.c_void_p()
    _chk(lib().dmrgx_truncate(kron.h, psi.ptr, LL(mstates), C.byref(l), C.byref(r)))
    return BasisTransformation(kron.ctx, l), BasisTransformation(kron.ctx, r)


class Wave:
    """EXTENSION (csrc/predict.cpp): this step's ground state with the growing side projected on its kept states;
    `apply` returns the start vector of the next step's eigen-solve, or None when the blocks do not chain up."""

    def __init__(self, kron, psi, bt_grown, grow_left=True):
        self.ctx = kron.ctx
        h = C.c_void_p()
        _chk(lib().dmrgx_wave_create(kron.h, psi.ptr, bt_grown.h, 1 if grow_left else 0, C.byref(h)))
        self.h = h

    def __del__(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            lib().dmrgx_wave_destroy(self.h)
            self.h = None

    def apply(self, bt_shrinking, site, kron_new):
        out = DeviceVector(self.ctx, kron_new.NumStates())
        ok = C.c_int(0)
        _chk(lib().dmrgx_wave_apply(self.h, bt_shrinking.h, site.h, kron_new.h, out.ptr, C.byref(ok)))
        return out if ok.value else None


def RotateOperators(enlarged, bt):
    """BlockOut.Initialize(nsites, BT.QN) + BlockOut.RotateOperators(BlockEnl, RotMatT) — src/DMRGBlock.cpp:677-823"""
    h = C.c_void_p()
    _chk(lib().dmrgx_rotate(enlarged.h, bt.h, C.byref(h)))
    return Block(enlarged.ctx, h)
