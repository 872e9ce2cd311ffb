"""ctypes loader for oracle/libecref.so (the C restatement of the reference's CPU path).
TEST INFRASTRUCTURE ONLY — see the header of ecref.c."""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(_HERE, "libecref.so")
_lib = None


def _host_tag():
    """-march=native binaries must be rebuilt on the machine that runs them: tag the build with the CPU flags."""
    import hashlib

    try:
        with open("/proc/cpuinfo") as f:
            flags = next((ln for ln in f if ln.startswith("flags")), "")
    except OSError:
        flags = ""
    return hashlib.sha1(flags.encode()).hexdigest()


def _make(lib_path, srcs, force=False):
    """(Re)build one oracle library with make when it is missing, older than its sources or built for another CPU."""
    tagf = lib_path + ".host"
    tag = _host_tag()
    srcs = [os.path.join(_HERE, s) for s in srcs]
    stale = (not os.path.exists(lib_path) or os.path.getmtime(lib_path) < max(os.path.getmtime(s) for s in srcs)
             or not os.path.exists(tagf) or open(tagf).read().strip() != tag)
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-B", os.path.basename(lib_path)], stdout=subprocess.DEVNULL)
        with open(tagf, "w") as f:
            f.write(tag)
    return lib_path


def build(force=False):
    return _make(LIB, ["ecref.c"], force)


def build_all(force=False):
    """Every oracle library with its CPU tag, so that later loads on this machine write nothing into the tree."""
    build(force)
    _make(LIB384, ["ecref_p384.c"], force)
    _make(LIBP, ["ecref_prime.c", "ecref_prime_impl.inc"], force)


def lib():
    global _lib
    if _lib is None:
        build()
        try:
            _lib = ctypes.CDLL(LIB)
            _lib.ecref_init()
        except OSError:
            build(force=True)
            _lib = ctypes.CDLL(LIB)
            _lib.ecref_init()
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        _lib.ecref_mul_batch.argtypes = [ctypes.c_int, sz, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_int]
        _lib.ecref_mul_gen_batch.argtypes = [ctypes.c_int, sz, vp, vp, vp, ctypes.c_int]
        _lib.ecref_mul_gen_add_batch.argtypes = [ctypes.c_int, sz, vp, vp, vp, vp, vp, vp, ctypes.c_int]
        _lib.ecref_lincomb.argtypes = [ctypes.c_int, sz, vp, vp, vp, vp, vp, ctypes.c_int]
        _lib.ecref_field_op.argtypes = [ctypes.c_int, ctypes.c_int, sz, vp, vp, vp]
        _lib.ecref_radix16.argtypes = [vp, ctypes.c_int, vp]
        _lib.ecref_wnaf.argtypes = [vp, sz, sz, ctypes.c_int, vp]
        _lib.ecref_wnaf.restype = ctypes.c_int
        _lib.ecref_glv.argtypes = [vp, vp, vp]
    return _lib


LIB384 = os.path.join(_HERE, "libecref384.so")
_lib384 = None


def lib384():
    """oracle/ecref_p384.c — the P-384 restatement (48-byte records)"""
    global _lib384
    if _lib384 is None:
        _make(LIB384, ["ecref_p384.c"])
        _lib384 = ctypes.CDLL(LIB384)
        _lib384.ecref384_init()
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        _lib384.ecref384_mul_batch.argtypes = [sz, vp, vp, vp, vp, vp, ctypes.c_int]
        _lib384.ecref384_mul_gen_batch.argtypes = [sz, vp, vp, vp, ctypes.c_int]
        _lib384.ecref384_lincomb.argtypes = [sz, vp, vp, vp, vp, vp, ctypes.c_int]
    return _lib384


LIBP = os.path.join(_HERE, "libecrefp.so")
_libp = None
# curves served by oracle/ecref_prime.c: id -> bytes per record (ids as in include/ecgpu.h)
EXT = {"sm2": 3, "bp256r1": 4, "bp256t1": 5, "bignp256": 6, "bp384r1": 7, "bp384t1": 8, "p224": 9, "p192": 10, "p521": 11}
EXT.update({v: v for v in list(EXT.values())})
EXT_NB = {3: 32, 4: 32, 5: 32, 6: 32, 7: 48, 8: 48, 9: 28, 10: 24, 11: 66}


def libp():
    """oracle/ecref_prime.c — the generic primeorder / Montgomery-field restatement (sm2, brainpool, bign, P-224, P-192)"""
    global _libp
    if _libp is None:
        _make(LIBP, ["ecref_prime.c", "ecref_prime_impl.inc"])
        _libp = ctypes.CDLL(LIBP)
        _libp.ecrefp_init()
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        _libp.ecrefp_mul_batch.argtypes = [ctypes.c_int, sz, vp, vp, vp, vp, vp, ctypes.c_int]
        _libp.ecrefp_mul_gen_batch.argtypes = [ctypes.c_int, sz, vp, vp, vp, ctypes.c_int]
        _libp.ecrefp_lincomb.argtypes = [ctypes.c_int, sz, vp, vp, vp, vp, vp, ctypes.c_int]
    return _libp


def _p(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else ctypes.c_void_p(0)


CURVE = {"k256": 0, "p256": 1, 0: 0, 1: 1}


def mul_batch(curve, k, pxy, pinf=None, nthreads=1, variant=0):
    k = np.ascontiguousarray(k, np.uint8).reshape(-1)
    pxy = np.ascontiguousarray(pxy, np.uint8).reshape(-1)
    if pinf is not None:
        pinf = np.ascontiguousarray(pinf, np.uint8).reshape(-1)
    if curve in EXT:
        cid = EXT[curve]
        nb = EXT_NB[cid]
        n = k.size // nb
        oxy = np.zeros(2 * nb * n, np.uint8)
        oinf = np.zeros(n, np.uint8)
        rc = libp().ecrefp_mul_batch(cid, n, _p(k), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads)
        if rc:
            raise ValueError(f"ecrefp_mul_batch rc={rc}")
        return oxy.reshape(n, 2 * nb), oinf
    if curve in ("p384", 2):
        n = k.size // 48
        oxy = np.zeros(96 * n, np.uint8)
        oinf = np.zeros(n, np.uint8)
        rc = lib384().ecref384_mul_batch(n, _p(k), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads)
        if rc:
            raise ValueError(f"ecref384_mul_batch rc={rc}")
        return oxy.reshape(n, 96), oinf
    n = k.size // 32
    oxy = np.zeros(64 * n, np.uint8)
    oinf = np.zeros(n, np.uint8)
    rc = lib().ecref_mul_batch(CURVE[curve], n, _p(k), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads, variant)
    if rc:
        raise ValueError(f"ecref_mul_batch rc={rc}")
    return oxy.reshape(n, 64), oinf


def mul_gen_batch(curve, k, nthreads=1):
    k = np.ascontiguousarray(k, np.uint8).reshape(-1)
    if curve in EXT:
        cid = EXT[curve]
        nb = EXT_NB[cid]
        n = k.size // nb
        oxy = np.zeros(2 * nb * n, np.uint8)
        oinf = np.zeros(n, np.uint8)
        rc = libp().ecrefp_mul_gen_batch(cid, n, _p(k), _p(oxy), _p(oinf), nthreads)
        if rc:
            raise ValueError(f"ecrefp_mul_gen_batch rc={rc}")
        return oxy.reshape(n, 2 * nb), oinf
    if curve in ("p384", 2):
        n = k.size // 48
        oxy = np.zeros(96 * n, np.uint8)
        oinf = np.zeros(n, np.uint8)
        rc = lib384().ecref384_mul_gen_batch(n, _p(k), _p(oxy), _p(oinf), nthreads)
        if rc:
            raise ValueError(f"ecref384_mul_gen_batch rc={rc}")
        return oxy.reshape(n, 96), oinf
    n = k.size // 32
    oxy = np.zeros(64 * n, np.uint8)
    oinf = np.zeros(n, np.uint8)
    rc = lib().ecref_mul_gen_batch(CURVE[curve], n, _p(k), _p(oxy), _p(oinf), nthreads)
    if rc:
        raise ValueError(f"ecref_mul_gen_batch rc={rc}")
    return oxy.reshape(n, 64), oinf


def mul_gen_add_batch(curve, a, b, pxy, pinf=None, nthreads=1):
    a = np.ascontiguousarray(a, np.uint8).reshape(-1)
    b = np.ascontiguousarray(b, np.uint8).reshape(-1)
    n = a.size // 32
    pxy = np.ascontiguousarray(pxy, np.uint8).reshape(-1)
    if pinf is not None:
        pinf = np.ascontiguousarray(pinf, np.uint8).reshape(-1)
    oxy = np.zeros(64 * n, np.uint8)
    oinf = np.zeros(n, np.uint8)
    rc = lib().ecref_mul_gen_add_batch(CURVE[curve], n, _p(a), _p(b), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads)
    if rc:
        raise ValueError(f"ecref_mul_gen_add_batch rc={rc}")
    return oxy.reshape(n, 64), oinf


def lincomb(curve, k, pxy, pinf=None, nthreads=1):
    k = np.ascontiguousarray(k, np.uint8).reshape(-1)
    pxy = np.ascontiguousarray(pxy, np.uint8).reshape(-1)
    if pinf is not None:
        pinf = np.ascontiguousarray(pinf, np.uint8).reshape(-1)
    if curve in EXT:
        cid = EXT[curve]
        nb = EXT_NB[cid]
        n = k.size // nb
        oxy = np.zeros(2 * nb, np.uint8)
        oinf = np.zeros(1, np.uint8)
        rc = libp().ecrefp_lincomb(cid, n, _p(k), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads)
        if rc:
            raise ValueError(f"ecrefp_lincomb rc={rc}")
        return oxy, int(oinf[0])
    if curve in ("p384", 2):
        n = k.size // 48
        oxy = np.zeros(96, np.uint8)
        oinf = np.zeros(1, np.uint8)
        rc = lib384().ecref384_lincomb(n, _p(k), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads)
        if rc:
            raise ValueError(f"ecref384_lincomb rc={rc}")
        return oxy, int(oinf[0])
    n = k.size // 32
    oxy = np.zeros(64, np.uint8)
    oinf = np.zeros(1, np.uint8)
    rc = lib().ecref_lincomb(CURVE[curve], n, _p(k), _p(pxy), _p(pinf), _p(oxy), _p(oinf), nthreads)
    if rc:
        raise ValueError(f"ecref_lincomb rc={rc}")
    return oxy, int(oinf[0])


def field_op(curve, op, a, b=None):
    a = np.ascontiguousarray(a, np.uint8).reshape(-1)
    n = a.size // 32
    if b is not None:
        b = np.ascontiguousarray(b, np.uint8).reshape(-1)
    out = np.zeros(32 * n, np.uint8)
    lib().ecref_field_op(CURVE[curve], op, n, _p(a), _p(b), _p(out))
    return out.reshape(n, 32)


def radix16(k_be: bytes, nd: int):
    kb = np.frombuffer(k_be, np.uint8).copy()
    out = np.zeros(nd, np.int8)
    lib().ecref_radix16(_p(kb), nd, _p(out))
    return out


def wnaf(le: bytes, bit_len: int, window: int):
    b = np.frombuffer(le, np.uint8).copy()
    out = np.zeros(bit_len + 8, np.int8)
    n = lib().ecref_wnaf(_p(b), len(le), bit_len, window, _p(out))
    return out[:n]


def glv(k: int):
    kb = np.frombuffer(k.to_bytes(32, "big"), np.uint8).copy()
    r1 = np.zeros(32, np.uint8)
    r2 = np.zeros(32, np.uint8)
    lib().ecref_glv(_p(kb), _p(r1), _p(r2))
    return int.from_bytes(r1.tobytes(), "big"), int.from_bytes(r2.tobytes(), "big")
