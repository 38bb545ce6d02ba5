"""The harness of the device-kernel tests: a ctypes backend over a test-only kernel shim (tests/devcheck/*.cpp), guard-banded
buffers and the extended-precision summation bound.  The conventions are argued in the docstring of test_device_kernels.py."""
import ctypes as C
import zlib

import numpy as np

U = 2.0 ** -53
LD = np.longdouble
SENT = np.uint64(0xC3D5A5A55A5A0F0F)   # output guard / gap sentinel (a finite double no kernel here produces)
MIN_GUARD = 512                          # 4 KiB of doubles


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
