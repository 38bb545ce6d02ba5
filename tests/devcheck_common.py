"""The harness of the device-kernel tests: a ctypes backend over a test-only kernel shim (tests/devcheck/*.cpp), guard-banded
buffers, the extended-precision summation bound, the record layouts of run_spmm and the input families of the eigensolver
tests.  The conventions are argued in the docstring of test_device_kernels.py."""
import ctypes as C
import os
import subprocess
import zlib

import numpy as np

U = 2.0 ** -53
LD = np.longdouble
SENT = np.uint64(0xC3D5A5A55A5A0F0F)   # output guard / gap sentinel (a finite double no kernel here produces)
MIN_GUARD = 512                          # 4 KiB of doubles

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dmrg.x_b200", "csrc")
LIBS = {"host": os.path.join(ROOT, "tests", "devcheck", "libdevcheck_host.so"),
        "cuda": os.path.join(ROOT, "tests", "devcheck", "libdevcheck_cuda.so")}
# DMRGX_DEVCHECK_CUDA: run the cuda flavour against another build of the shim (for example over a modified dev_cuda.cu)
CUDA_OVERRIDE = os.environ.get("DMRGX_DEVCHECK_CUDA")

# csrc/dev.h: the records of run_spmm (element offsets where the product has pointers: see tests/devcheck/devcheck.cpp)
SP_ROWS, SP_MAX_NR = 4, 3072
SP_TILE = np.dtype([("off", "<i8"), ("nR", "<i4"), ("nrows", "<i4"), ("a_begin", "<i4"), ("a_count", "<i4"), ("s_begin", "<i4"), ("s_count", "<i4"),
                    ("b_begin", "<i4"), ("b_count", "<i4"), ("pad", "<i4", 6)])
SP_ASLOT = np.dtype([("src", "<i8", SP_ROWS), ("w", "<f8", SP_ROWS)])
SP_SSLOT = np.dtype([("roff", "<i4", SP_ROWS), ("pad", "<i4", SP_ROWS), ("w", "<f8", SP_ROWS)])
SP_BSLOT = np.dtype([("ecol", "<i8"), ("eval", "<i8"), ("W", "<i4"), ("ld", "<i4"), ("all_in", "<i4"), ("pad", "<i4"), ("roff", "<i4", SP_ROWS),
                     ("src", "<i8", SP_ROWS), ("w", "<f8", SP_ROWS)])
assert SP_TILE.itemsize == 64 and SP_ASLOT.itemsize == 64 and SP_SSLOT.itemsize == 64 and SP_BSLOT.itemsize == 112


def lib_path(name):
    """the shim over the host emulation or over the product's sm_100a object, built on first use"""
    if name == "cuda" and CUDA_OVERRIDE:
        return CUDA_OVERRIDE
    path = LIBS[name]
    if not os.path.exists(path):
        subprocess.check_call(["make", "-s", "-C", CSRC, "devcheck-" + name])
    return path


class Backend:
    def __init__(self, name, path):
        self.name = name
        self.lib = C.CDLL(path)
        self.lib.dc_error.restype = C.c_char_p

    def __call__(self, fn, *args):
        conv = []
        for a in args:
            if isinstance(a, np.ndarray):
                assert a.flags.c_contiguous
                conv.append(C.c_void_p(a.ctypes.data))
            elif a is None:
                conv.append(C.c_void_p(None))
            elif isinstance(a, float):
                conv.append(C.c_double(a))
            elif isinstance(a, tuple):          # ("u64", value)
                conv.append(C.c_ulonglong(a[1]))
            else:
                conv.append(C.c_longlong(int(a)))
        return getattr(self.lib, fn)(*conv)

    def ok(self, fn, *args):
        rc = self(fn, *args)
        assert rc == 0, "%s: %s" % (fn, self.error())

    def refused(self, fn, *args):
        rc = self(fn, *args)
        assert rc != 0, "%s was not refused" % fn
        return self.error()

    def error(self):
        return self.lib.dc_error().decode()


def guard_for(ld=0):
    g = max(MIN_GUARD, int(ld))
    return g + (g & 1)


def wrap(payload, g, fill="nan"):
    """[guard | payload | guard]; fill: 'nan' (operands) or 'sent' (outputs)"""
    payload = np.ascontiguousarray(payload)
    full = np.empty(payload.size + 2 * g, payload.dtype)
    if fill == "sent":
        full.view(np.uint64)[:] = SENT
    elif payload.dtype == np.float64:
        full[:] = np.nan
    else:
        full[:] = 0
    full[g:g + payload.size] = payload.ravel()
    return full


def sentinel(n, g):
    full = np.empty(n + 2 * g)
    full.view(np.uint64)[:] = SENT
    return full


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def assert_guards(full, g, what="output"):
    assert (bits(full[:g]) == SENT).all() and (bits(full[-g:]) == SENT).all(), "%s guard overwritten" % what


def assert_unchanged(after, before, sel, what):
    assert (bits(after[sel]) == bits(before[sel])).all(), "%s changed where it must not" % what


def assert_bound(got, ref, absref, N, what):
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, LD)
    bound = (np.asarray(N, LD) + 2) * LD(U) * np.asarray(absref, LD)
    err = np.abs(got.astype(LD) - ref)
    bad = ~(err <= bound)
    if bad.any():
        i = np.flatnonzero(bad.ravel())[0]
        raise AssertionError("%s: %d elements outside (N+2)·u·Σ|terms|; first at flat %d: got %r ref %r bound %r"
                             % (what, int(bad.sum()), i, float(got.ravel()[i]), float(ref.ravel()[i]), float(np.broadcast_to(bound, got.shape).ravel()[i])))


def rng_for(*key):
    return np.random.default_rng([zlib.crc32(str(k).encode()) for k in key])


# ---------------------------------------------------------------------------------------------------------------------
#  inputs of the eigensolver tests (test_sparse_eig_kernels.py through the shim, test_gpu_parity.py through the C ABI)
# ---------------------------------------------------------------------------------------------------------------------
def rho_like(rng, n):
    k = max(1, (2 * n) // 3)                                   # rank-deficient like rho_L of a wide psi block
    X = rng.standard_normal((n, k)) * np.exp(-0.35 * np.arange(k))[None, :]
    R = X @ X.T
    return R / np.trace(R)


def with_spectrum(rng, lam):
    Q, _ = np.linalg.qr(rng.standard_normal((len(lam), len(lam))))
    R = (Q * lam[None, :]) @ Q.T
    return (R + R.T) / 2


def eig_inputs(case):
    """rho-like blocks at the listed sizes, or the named input family"""
    rng = np.random.default_rng(12)
    if isinstance(case, list):
        return [rho_like(rng, n) for n in case]
    if case == "multiplets":   # exact multiplicities 2-8, as SU(2)-symmetric rho blocks have, on both solver paths
        out = []
        for n in (36, 150):
            lam = np.concatenate([np.full(mult, v) for mult, v in zip(np.resize(np.arange(2, 9), n), np.exp(-rng.uniform(0, 20, n)))])[:n]
            out.append(with_spectrum(rng, np.sort(lam)[::-1]))
        return out
    if case == "diagonal":     # already converged
        return [np.diag(rng.standard_normal(n)) for n in (1, 30, 64, 100, 193)]
    if case == "zero":
        return [np.zeros((n, n)) for n in (1, 10, 64, 70, 129)]
    if case == "indefinite":   # padding coordinates must keep their trailing positions among negative eigenvalues
        return [with_spectrum(rng, rng.standard_normal(n)) for n in (50, 65, 130, 193)]
    if case == "negative-definite":
        return [-rho_like(rng, n) - 0.1 * np.eye(n) for n in (64, 65, 129, 192)]
    if case == "batch-300":
        return [rho_like(rng, int(n)) for n in rng.integers(1, 65, 300)]
    raise ValueError(case)
