"""ecgpu — Python (ctypes) host-side mirror of the reference's operator surface over libecgpu.so.

The shared library is the product; this module is the thinnest possible binding used by tests/ and
bench.py.  It mirrors the reference's names for the hot path:

    Engine.mul_batch(curve, k, P)              ProjectivePoint * Scalar over a batch     (k256/src/arithmetic/mul.rs:236-295)
    Engine.mul_by_generator(curve, k)          ProjectivePoint::mul_by_generator         (mul.rs:180-232)
    Engine.lincomb(curve, k, P)                LinearCombination::lincomb                (mul.rs:66-175)
    Engine.mul_by_generator_and_mul_add(...)   MulByGeneratorVartime::..._and_mul_add    (mul.rs:303-310)
    Engine.batch_normalize(curve, XYZ)         BatchNormalize::batch_normalize           (projective.rs:345-391)
    Engine.field_op(curve, op, a, b)           FieldElement add/sub/neg/mul/square/invert
    Engine.sm2pke_encrypt / sm2pke_decrypt     sm2 EncryptingKey::encrypt / DecryptingKey::decrypt over a batch
                                               (`*_vartime` on a ctx without ECG_FLAG_CONSTTIME)

Buffers are numpy uint8 arrays (host mode) or raw device pointers (device mode, ECG_FLAG_DEVICE_PTRS).
There is NO CPU fallback: if libecgpu.so is missing, or no CUDA device is present, construction raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libecgpu.so")

SECP256K1 = 0
NISTP256 = 1
NISTP384 = 2
SM2, BP256R1, BP256T1, BIGNP256, BP384R1, BP384T1, NISTP224, NISTP192, NISTP521 = 3, 4, 5, 6, 7, 8, 9, 10, 11
CURVE_IDS = {"k256": SECP256K1, "secp256k1": SECP256K1, "p256": NISTP256, "nistp256": NISTP256, "p384": NISTP384, "nistp384": NISTP384,
             "sm2": SM2, "bp256r1": BP256R1, "brainpoolp256r1": BP256R1, "bp256t1": BP256T1, "brainpoolp256t1": BP256T1,
             "bignp256": BIGNP256, "bp384r1": BP384R1, "brainpoolp384r1": BP384R1, "bp384t1": BP384T1, "brainpoolp384t1": BP384T1,
             "p224": NISTP224, "nistp224": NISTP224, "p192": NISTP192, "nistp192": NISTP192, "p521": NISTP521, "nistp521": NISTP521}
CURVE_IDS.update({i: i for i in range(12)})
# bytes per scalar / coordinate at the ABI (include/ecgpu.h)
FBYTES = {SECP256K1: 32, NISTP256: 32, NISTP384: 48, SM2: 32, BP256R1: 32, BP256T1: 32, BIGNP256: 32, BP384R1: 48, BP384T1: 48,
          NISTP224: 28, NISTP192: 24, NISTP521: 66}
# bign-curve256v1 records are little-endian (the reference's byte order for that curve); every other curve is big-endian
LITTLE_ENDIAN = {BIGNP256}

ECG_OK, ECG_EINVAL, ECG_ESCALAR_RANGE, ECG_ENOT_ON_CURVE, ECG_ECUDA, ECG_ENCCL, ECG_ENOMEM = range(7)
FLAG_DEVICE_PTRS = 1
FLAG_ZEROIZE = 2
FLAG_CONSTTIME = 4  # scalar-independent table selects / sign folding, k*G through the variable-base routine, per-term lincomb
FOP = {"add": 0, "sub": 1, "neg": 2, "mul": 3, "sqr": 4, "inv": 5}

EXPORTS = [
    "ecg_ctx_create", "ecg_ctx_destroy", "ecg_last_error", "ecg_last_error_index", "ecg_ctx_set_stream",
    "ecg_mul_batch", "ecg_mul_gen_batch", "ecg_lincomb", "ecg_lincomb_partial", "ecg_point_sum",
    "ecg_mul_gen_add_batch", "ecg_batch_normalize", "ecg_field_op_batch", "ecg_microbench",
    "ecg_kernel_launches", "ecg_version", "ecg_timing_enable", "ecg_timing_read",
    "ecg_schnorr_verify_batch", "ecg_ecdsa_verify_batch", "ecg_decompress_batch",
    "ecg_batch_normalize_hom", "ecg_mul_batch_x", "ecg_field_sqrt_batch",
    "ecg_hash_to_curve_batch", "ecg_hash_to_scalar_batch", "ecg_sm2dsa_verify_batch", "ecg_ecdsa_recover_batch",
    "ecg_sm2pke_encrypt_batch", "ecg_sm2pke_decrypt_batch",
]
# SM2 public-key encryption ciphertext layouts (sm2/src/pke.rs Mode; C1C3C2 is the reference's default)
SM2PKE_MODES = {"c1c3c2": 0, "c1c2c3": 1, 0: 0, 1: 1}


class EcgError(RuntimeError):
    def __init__(self, code: int, msg: str, index: int = -1):
        super().__init__(f"ecgpu error {code}: {msg}" + (f" (first offending index {index})" if index >= 0 else ""))
        self.code = code
        self.index = index


class ScalarRangeError(EcgError):
    """Scalar::from_repr returned None in the reference (k >= n)."""


class NotOnCurveError(EcgError):
    """AffinePoint::from_coordinates returned None in the reference."""


_lib = None


def load_library(path: Optional[str] = None) -> ctypes.CDLL:
    """dlopen libecgpu.so (fails loudly if it has not been built: run `python -c 'import __graft_entry__ as g; g.build()'`)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FileNotFoundError(f"{p} not found: the CUDA extension is not built (no CPU fallback exists)")
    lib = ctypes.CDLL(p)
    vp, sz, u8p = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p
    lib.ecg_ctx_create.argtypes = [ctypes.POINTER(ctypes.c_int), ctypes.c_int, ctypes.c_uint, ctypes.POINTER(vp)]
    lib.ecg_ctx_create.restype = ctypes.c_int
    lib.ecg_ctx_destroy.argtypes = [vp]
    lib.ecg_ctx_destroy.restype = None
    lib.ecg_last_error.argtypes = [vp]
    lib.ecg_last_error.restype = ctypes.c_char_p
    lib.ecg_last_error_index.argtypes = [vp]
    lib.ecg_last_error_index.restype = sz
    lib.ecg_ctx_set_stream.argtypes = [vp, vp]
    lib.ecg_ctx_set_stream.restype = ctypes.c_int
    lib.ecg_mul_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, u8p, u8p]
    lib.ecg_mul_batch.restype = ctypes.c_int
    lib.ecg_mul_gen_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p]
    lib.ecg_mul_gen_batch.restype = ctypes.c_int
    lib.ecg_lincomb.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, u8p, u8p]
    lib.ecg_lincomb.restype = ctypes.c_int
    lib.ecg_lincomb_partial.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, u8p]
    lib.ecg_lincomb_partial.restype = ctypes.c_int
    lib.ecg_point_sum.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p]
    lib.ecg_point_sum.restype = ctypes.c_int
    lib.ecg_mul_gen_add_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, u8p, u8p, u8p]
    lib.ecg_mul_gen_add_batch.restype = ctypes.c_int
    lib.ecg_batch_normalize.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p]
    lib.ecg_batch_normalize.restype = ctypes.c_int
    lib.ecg_field_op_batch.argtypes = [vp, ctypes.c_int, ctypes.c_int, sz, u8p, u8p, u8p]
    lib.ecg_field_op_batch.restype = ctypes.c_int
    lib.ecg_microbench.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]
    lib.ecg_microbench.restype = ctypes.c_int
    lib.ecg_kernel_launches.argtypes = [vp]
    lib.ecg_kernel_launches.restype = ctypes.c_uint64
    lib.ecg_timing_enable.argtypes = [vp, ctypes.c_int]
    lib.ecg_timing_enable.restype = ctypes.c_int
    lib.ecg_timing_read.argtypes = [vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]
    lib.ecg_timing_read.restype = ctypes.c_int
    lib.ecg_schnorr_verify_batch.argtypes = [vp, sz, u8p, u8p, u8p, u8p]
    lib.ecg_schnorr_verify_batch.restype = ctypes.c_int
    lib.ecg_ecdsa_verify_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, ctypes.c_int, u8p]
    lib.ecg_ecdsa_verify_batch.restype = ctypes.c_int
    lib.ecg_sm2dsa_verify_batch.argtypes = [vp, sz, u8p, u8p, u8p, u8p]
    lib.ecg_ecdsa_recover_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, ctypes.c_int, u8p, u8p]
    lib.ecg_ecdsa_recover_batch.restype = ctypes.c_int
    lib.ecg_sm2dsa_verify_batch.restype = ctypes.c_int
    lib.ecg_decompress_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, u8p]
    lib.ecg_decompress_batch.restype = ctypes.c_int
    lib.ecg_batch_normalize_hom.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p]
    lib.ecg_batch_normalize_hom.restype = ctypes.c_int
    lib.ecg_mul_batch_x.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, u8p, u8p]
    lib.ecg_mul_batch_x.restype = ctypes.c_int
    lib.ecg_field_sqrt_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p]
    lib.ecg_field_sqrt_batch.restype = ctypes.c_int
    lib.ecg_hash_to_curve_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, sz, ctypes.c_int, u8p, u8p]
    lib.ecg_hash_to_curve_batch.restype = ctypes.c_int
    lib.ecg_hash_to_scalar_batch.argtypes = [vp, ctypes.c_int, sz, u8p, u8p, u8p, sz, u8p]
    lib.ecg_hash_to_scalar_batch.restype = ctypes.c_int
    lib.ecg_sm2pke_encrypt_batch.argtypes = [vp, sz, u8p, u8p, u8p, u8p, ctypes.c_int, ctypes.c_int, u8p, u8p]
    lib.ecg_sm2pke_encrypt_batch.restype = ctypes.c_int
    lib.ecg_sm2pke_decrypt_batch.argtypes = [vp, sz, u8p, u8p, u8p, ctypes.c_int, u8p, u8p, u8p]
    lib.ecg_sm2pke_decrypt_batch.restype = ctypes.c_int
    lib.ecg_version.argtypes = []
    lib.ecg_version.restype = ctypes.c_char_p
    if path is None:
        _lib = lib
    return lib


def _u8(a, nbytes: int, name: str) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    if a.size != nbytes:
        raise ValueError(f"{name}: expected {nbytes} bytes, got {a.size}")
    return a


def _out(a, nbytes: int, name: str) -> np.ndarray:
    """a caller-supplied output array is written in place by the library: it must be exactly what the ABI expects"""
    if a is None:
        return np.empty(nbytes, np.uint8)
    if not (isinstance(a, np.ndarray) and a.dtype == np.uint8 and a.flags["C_CONTIGUOUS"] and a.flags["WRITEABLE"] and a.size == nbytes):
        raise ValueError(f"{name}: expected a writable C-contiguous uint8 array of {nbytes} bytes")
    return a


def _ptr(a) -> ctypes.c_void_p:
    if a is None:
        return ctypes.c_void_p(0)
    if isinstance(a, np.ndarray):
        return ctypes.c_void_p(a.ctypes.data)
    return ctypes.c_void_p(int(a))  # raw device pointer


class Engine:
    """One ecg_ctx.  `devices=[0]` host-pointer mode by default; `device_ptrs=True` takes raw CUDA pointers."""

    def __init__(self, devices: Optional[Sequence[int]] = None, device_ptrs: bool = False, zeroize: bool = False, consttime: bool = False):
        self.lib = load_library()
        devs = list(devices) if devices else [0]
        arr = (ctypes.c_int * len(devs))(*devs)
        self._ctx = ctypes.c_void_p(0)
        self.device_ptrs = device_ptrs
        self.consttime = consttime
        flags = (FLAG_DEVICE_PTRS if device_ptrs else 0) | (FLAG_ZEROIZE if zeroize else 0) | (FLAG_CONSTTIME if consttime else 0)
        rc = self.lib.ecg_ctx_create(arr, len(devs), flags, ctypes.byref(self._ctx))
        if rc != ECG_OK:
            raise EcgError(rc, "ecg_ctx_create failed (is a CUDA device visible? there is no CPU fallback)")

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self.lib.ecg_ctx_destroy(self._ctx)
            self._ctx = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc == ECG_OK:
            return
        msg = (self.lib.ecg_last_error(self._ctx) or b"").decode()
        idx = int(self.lib.ecg_last_error_index(self._ctx))
        if idx == 2**64 - 1:
            idx = -1
        if rc == ECG_ESCALAR_RANGE:
            raise ScalarRangeError(rc, msg, idx)
        if rc == ECG_ENOT_ON_CURVE:
            raise NotOnCurveError(rc, msg, idx)
        raise EcgError(rc, msg, idx)

    def set_stream(self, cuda_stream: int):
        """Run this ctx's work on the caller's CUDA stream (e.g. `torch.cuda.current_stream().cuda_stream`).  PyTorch's
        default stream has the handle 0, which the C ABI reads as "back to the ctx-owned stream": it is passed as
        cudaStreamLegacy (1), the explicit name of the same stream, so that the library's kernels are ordered with the
        producer of their inputs (a collective, a copy) instead of racing on a separate non-blocking stream."""
        if cuda_stream == 0:
            cuda_stream = 1  # cudaStreamLegacy
        self._check(self.lib.ecg_ctx_set_stream(self._ctx, ctypes.c_void_p(cuda_stream)))

    def reset_stream(self):
        self._check(self.lib.ecg_ctx_set_stream(self._ctx, ctypes.c_void_p(0)))

    @property
    def kernel_launches(self) -> int:
        return int(self.lib.ecg_kernel_launches(self._ctx))

    # ---- host-pointer API (numpy) ----
    def mul_batch(self, curve, k, P_xy, P_inf=None, out_xy=None, out_inf=None):
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(k).size // fb
        k = _u8(k, fb * n, "k")
        P_xy = _u8(P_xy, 2 * fb * n, "P_xy")
        if P_inf is not None:
            P_inf = _u8(P_inf, n, "P_inf")
        out_xy = _out(out_xy, 2 * fb * n, "out_xy")
        out_inf = _out(out_inf, n, "out_inf")
        self._check(self.lib.ecg_mul_batch(self._ctx, c, n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out_xy), _ptr(out_inf)))
        return out_xy.reshape(n, 2 * fb), out_inf

    def mul_by_generator(self, curve, k, out_xy=None, out_inf=None):
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(k).size // fb
        k = _u8(k, fb * n, "k")
        out_xy = _out(out_xy, 2 * fb * n, "out_xy")
        out_inf = _out(out_inf, n, "out_inf")
        self._check(self.lib.ecg_mul_gen_batch(self._ctx, c, n, _ptr(k), _ptr(out_xy), _ptr(out_inf)))
        return out_xy.reshape(n, 2 * fb), out_inf

    def mul_batch_x(self, curve, k, P_xy, P_inf=None):
        """x coordinate of k[i] * P[i] only (ecg_mul_batch_x) -> (x n x 32, inf)"""
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(k).size // fb
        k = _u8(k, fb * n, "k")
        P_xy = _u8(P_xy, 2 * fb * n, "P_xy")
        if P_inf is not None:
            P_inf = _u8(P_inf, n, "P_inf")
        out_x = np.empty(fb * n, np.uint8)
        out_inf = np.empty(n, np.uint8)
        self._check(self.lib.ecg_mul_batch_x(self._ctx, c, n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out_x), _ptr(out_inf)))
        return out_x.reshape(n, fb), out_inf

    def diffie_hellman_vartime(self, curve, secret_k, public_xy):
        """ECDH batch: x-coordinate of k[i] * P[i] (k256/src/ecdh.rs:46-60 `diffie_hellman`: `(public * secret).to_affine().x`).

        VARIABLE TIME in the secret: the kernels index window tables by scalar digits and branch on exceptional cases
        (INTEGRATION.md "constant time"); the reference's `diffie_hellman` is constant time.  Hence the name: use it
        only where timing of the device is not observable by an adversary, with an Engine(zeroize=True) so the staged
        scalars and tables are cleared after the call.  As in the reference, the inputs are a NonZeroScalar and a
        PublicKey: a zero scalar or an identity result is refused (ValueError) instead of yielding an all-zero secret."""
        fb = FBYTES[CURVE_IDS[curve]]
        n = np.asarray(secret_k).size // fb
        kk = _u8(secret_k, fb * n, "secret_k").reshape(n, fb)
        if n and not kk.any(axis=1).all():
            raise ValueError("diffie_hellman_vartime: zero secret scalar (the reference takes a NonZeroScalar)")
        out_x, out_inf = self.mul_batch_x(curve, kk, public_xy, None)
        if out_inf.any():
            raise ValueError("diffie_hellman_vartime: identity shared point")
        return out_x

    def lincomb(self, curve, k, P_xy, P_inf=None):
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(k).size // fb
        k = _u8(k, fb * n, "k")
        P_xy = _u8(P_xy, 2 * fb * n, "P_xy")
        if P_inf is not None:
            P_inf = _u8(P_inf, n, "P_inf")
        out_xy = np.zeros(2 * fb, np.uint8)
        out_inf = np.zeros(1, np.uint8)
        self._check(self.lib.ecg_lincomb(self._ctx, c, n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out_xy), _ptr(out_inf)))
        return out_xy, int(out_inf[0])

    def lincomb_partial(self, curve, k, P_xy, P_inf=None):
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(k).size // fb
        k = _u8(k, fb * n, "k")
        P_xy = _u8(P_xy, 2 * fb * n, "P_xy")
        if P_inf is not None:
            P_inf = _u8(P_inf, n, "P_inf")
        out = np.zeros(3 * fb, np.uint8)
        self._check(self.lib.ecg_lincomb_partial(self._ctx, c, n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out)))
        return out

    def point_sum(self, curve, xyz):
        c = CURVE_IDS[curve]
        xyz = np.ascontiguousarray(xyz, dtype=np.uint8).reshape(-1)
        m = xyz.size // (3 * FBYTES[c])
        out_xy = np.zeros(2 * FBYTES[c], np.uint8)
        out_inf = np.zeros(1, np.uint8)
        self._check(self.lib.ecg_point_sum(self._ctx, c, m, _ptr(xyz), _ptr(out_xy), _ptr(out_inf)))
        return out_xy, int(out_inf[0])

    def mul_by_generator_and_mul_add(self, curve, a, b, P_xy, P_inf=None):
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(a).size // fb
        a = _u8(a, fb * n, "a")
        b = _u8(b, fb * n, "b")
        P_xy = _u8(P_xy, 2 * fb * n, "P_xy")
        if P_inf is not None:
            P_inf = _u8(P_inf, n, "P_inf")
        out_xy = np.empty(2 * fb * n, np.uint8)
        out_inf = np.empty(n, np.uint8)
        self._check(self.lib.ecg_mul_gen_add_batch(self._ctx, c, n, _ptr(a), _ptr(b), _ptr(P_xy), _ptr(P_inf), _ptr(out_xy), _ptr(out_inf)))
        return out_xy.reshape(n, 2 * fb), out_inf

    @staticmethod
    def _pack_messages(msgs):
        """list of bytes -> (concatenated uint8 array, n + 1 uint64 offsets)"""
        offs = np.zeros(len(msgs) + 1, np.uint64)
        if len(msgs):
            offs[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
        data = np.frombuffer(b"".join(bytes(m) for m in msgs), np.uint8).copy() if offs[-1] else np.zeros(1, np.uint8)
        return data, offs

    def hash_to_curve(self, curve, msgs, dst: bytes, nonuniform: bool = False):
        """GroupDigest::hash_from_bytes / encode_from_bytes over a batch of messages (hash2curve/src/group_digest.rs:88-118)
        -> (xy n x 64, inf)"""
        data, offs = self._pack_messages(msgs)
        return self.hash_to_curve_packed(curve, data, offs, dst, nonuniform)

    def hash_to_curve_packed(self, curve, data, offsets, dst: bytes, nonuniform: bool = False, out_xy=None, out_inf=None):
        """the same over messages already laid out as the C ABI takes them: `data` = the messages back to back (uint8),
        `offsets` = n + 1 uint64 byte offsets (message i = data[offsets[i]:offsets[i + 1]])"""
        c = CURVE_IDS[curve]
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offs.size - 1
        if n < 0 or (n >= 0 and offs.size and int(offs[-1]) > np.asarray(data).size):
            raise ValueError("offsets: n + 1 ascending byte offsets into data")
        data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        if data.size == 0:
            data = np.zeros(1, np.uint8)
        d = np.frombuffer(bytes(dst), np.uint8).copy() if len(dst) else np.zeros(1, np.uint8)
        fb = FBYTES[c]
        out_xy = _out(out_xy, 2 * fb * n, "out_xy")
        out_inf = _out(out_inf, n, "out_inf")
        self._check(self.lib.ecg_hash_to_curve_batch(self._ctx, c, n, _ptr(data), _ptr(offs), _ptr(d), len(dst), 1 if nonuniform else 0,
                                                     _ptr(out_xy), _ptr(out_inf)))
        return out_xy.reshape(n, 2 * fb), out_inf

    def encode_to_curve(self, curve, msgs, dst: bytes):
        return self.hash_to_curve(curve, msgs, dst, nonuniform=True)

    def hash_to_scalar(self, curve, msgs, dst: bytes):
        """hash2curve::hash_to_scalar over a batch (group_digest.rs:131-143) -> n x 32 big-endian scalars"""
        c = CURVE_IDS[curve]
        n = len(msgs)
        data, offs = self._pack_messages(msgs)
        d = np.frombuffer(bytes(dst), np.uint8).copy() if len(dst) else np.zeros(1, np.uint8)
        fb = FBYTES[c]
        out = np.empty(fb * n, np.uint8)
        self._check(self.lib.ecg_hash_to_scalar_batch(self._ctx, c, n, _ptr(data), _ptr(offs), _ptr(d), len(dst), _ptr(out)))
        return out.reshape(n, fb)

    def schnorr_verify_batch(self, pk_x, msg32, sig64):
        """BIP340: VerifyingKey::verify_raw over a batch (k256/src/schnorr/verifying.rs:76-99) -> uint8 flags"""
        n = np.asarray(pk_x).size // 32
        pk_x = _u8(pk_x, 32 * n, "pk_x")
        msg32 = _u8(msg32, 32 * n, "msg32")
        sig64 = _u8(sig64, 64 * n, "sig64")
        valid = np.zeros(n, np.uint8)
        self._check(self.lib.ecg_schnorr_verify_batch(self._ctx, n, _ptr(pk_x), _ptr(msg32), _ptr(sig64), _ptr(valid)))
        return valid

    def ecdsa_verify_batch(self, curve, z32, sig64, Q_xy, low_s_only=False):
        """ECDSA verify_prehash over a batch -> uint8 flags.  Records are FB bytes (the curve's FieldBytes): z = the prehash
        after bits2field, signature r || s, public key x || y."""
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(z32).size // fb
        z32 = _u8(z32, fb * n, "z")
        sig64 = _u8(sig64, 2 * fb * n, "sig")
        Q_xy = _u8(Q_xy, 2 * fb * n, "Q_xy")
        valid = np.zeros(n, np.uint8)
        self._check(self.lib.ecg_ecdsa_verify_batch(self._ctx, c, n, _ptr(z32), _ptr(sig64), _ptr(Q_xy), 1 if low_s_only else 0, _ptr(valid)))
        return valid

    def ecdsa_recover_batch(self, curve, z32, sig64, recid, low_s_only=False, out_xy=None, valid=None):
        """VerifyingKey::recover_from_prehash over a batch (secp256k1 / P-256) -> (Q_xy n x 64, valid): prehash, r || s, one
        RecoveryId byte (bit 0: y of R odd, bit 1: x of R = r + n) per signature"""
        c = CURVE_IDS[curve]
        n = np.asarray(recid).size
        z32 = _u8(z32, 32 * n, "z")
        sig64 = _u8(sig64, 64 * n, "sig")
        recid = _u8(recid, n, "recid")
        out_xy = _out(out_xy, 64 * n, "out_xy")
        valid = _out(valid, n, "valid")
        self._check(self.lib.ecg_ecdsa_recover_batch(self._ctx, c, n, _ptr(z32), _ptr(sig64), _ptr(recid), 1 if low_s_only else 0,
                                                     _ptr(out_xy), _ptr(valid)))
        return out_xy.reshape(n, 64), valid

    def sm2dsa_verify_batch(self, e32, sig64, Q_xy):
        """SM2DSA verify_prehash over a batch -> uint8 flags: e = SM3(Z_A || M) (32 bytes), signature r || s, public key x || y"""
        n = np.asarray(e32).size // 32
        e32 = _u8(e32, 32 * n, "e")
        sig64 = _u8(sig64, 64 * n, "sig")
        Q_xy = _u8(Q_xy, 64 * n, "Q_xy")
        valid = np.zeros(n, np.uint8)
        self._check(self.lib.ecg_sm2dsa_verify_batch(self._ctx, n, _ptr(e32), _ptr(sig64), _ptr(Q_xy), _ptr(valid)))
        return valid

    # ---- SM2 public-key encryption (ecg_sm2pke_{encrypt,decrypt}_batch; sm2/src/pke/{encrypting,decrypting}.rs) ----
    # Without ECG_FLAG_CONSTTIME the scalar multiplications by k and d run the variable-time kernels, so, as with
    # diffie_hellman_vartime, the methods of a default ctx carry the `_vartime` suffix; an Engine(consttime=True) serves
    # the plain names.  Engine(zeroize=True) scrubs d, k, the staged messages and plaintexts and (x2, y2) after each call.
    def _sm2pke_ct(self, name):
        if not self.consttime:
            raise ValueError(f"{name}: this Engine runs the variable-time kernels; create it with consttime=True or call {name}_vartime")

    @staticmethod
    def _broadcast(a, rec: int, n: int, name: str) -> np.ndarray:
        """one record (broadcast to all n elements) or n records of `rec` bytes"""
        a = np.ascontiguousarray(np.frombuffer(bytes(a), np.uint8) if isinstance(a, (bytes, bytearray)) else a, dtype=np.uint8).reshape(-1)
        if a.size == rec:
            return np.ascontiguousarray(np.broadcast_to(a, (n, rec))).reshape(-1) if n else np.zeros(rec, np.uint8)
        return _u8(a, rec * n, name)

    def sm2pke_encrypt_packed_vartime(self, data, offsets, k, Pb, mode="c1c3c2", compressed: bool = True):
        """SM2 encryption of messages laid out as the C ABI takes them (`data` back to back, n + 1 uint64 `offsets`), with
        the caller's ephemeral scalars k (n x 32 bytes) and the recipient key(s) Pb (64 bytes x || y, or n x 64)
        -> (out, out_offsets, status): ciphertext i = out[out_offsets[i]:out_offsets[i + 1]] (zero bytes unless status[i]
        = 1); status 0 = refused (k not in [1, n-1], Pb off the curve, empty message), 2 = all-zero KDF output: draw
        another k (the reference's retry loop, encrypting.rs:184-209)."""
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offs.size - 1
        data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        if n < 0 or int(offs[-1]) > data.size:
            raise ValueError("offsets: n + 1 non-decreasing byte offsets into data")
        if data.size == 0:
            data = np.zeros(1, np.uint8)
        k = _u8(k, 32 * n, "k")
        Pb = self._broadcast(Pb, 64, n, "Pb")
        ovh = 32 + (33 if compressed else 65)
        out_offs = (offs - offs[0]) + np.arange(n + 1, dtype=np.uint64) * np.uint64(ovh) if n >= 0 else offs
        out = np.zeros(max(int(out_offs[-1]), 1), np.uint8)
        status = np.zeros(n, np.uint8)
        self._check(self.lib.ecg_sm2pke_encrypt_batch(self._ctx, n, _ptr(data), _ptr(offs), _ptr(k), _ptr(Pb), SM2PKE_MODES[mode],
                                                      1 if compressed else 0, _ptr(out), _ptr(status)))
        return out[:int(out_offs[-1])], out_offs, status

    def sm2pke_decrypt_packed_vartime(self, data, offsets, d, mode="c1c3c2"):
        """SM2 decryption of packed ciphertexts (C1 in any SEC1 form the reference accepts) under the secret key(s) d
        (32 bytes, or n x 32) -> (out, pt_len, valid): plaintext i = out[offsets[i] - offsets[0]:][:pt_len[i]]"""
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = offs.size - 1
        data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        if n < 0 or int(offs[-1]) > data.size:
            raise ValueError("offsets: n + 1 non-decreasing byte offsets into data")
        if data.size == 0:
            data = np.zeros(1, np.uint8)
        d = self._broadcast(d, 32, n, "d")
        total = int(offs[-1] - offs[0]) if n > 0 else 0
        out = np.zeros(max(total, 1), np.uint8)
        pt_len = np.zeros(n, np.uint64)
        valid = np.zeros(n, np.uint8)
        self._check(self.lib.ecg_sm2pke_decrypt_batch(self._ctx, n, _ptr(data), _ptr(offs), _ptr(d), SM2PKE_MODES[mode], _ptr(out),
                                                      _ptr(pt_len), _ptr(valid)))
        return out[:total], pt_len, valid

    def sm2pke_encrypt_vartime(self, msgs, k, Pb, mode="c1c3c2", compressed: bool = True):
        """EncryptingKey::encrypt over a list of messages (sm2/src/pke/encrypting.rs:166-230, digest SM3) with the caller's k
        -> (ciphertexts, status): ciphertext i is bytes where status[i] = 1, else None"""
        data, offs = self._pack_messages(msgs)
        out, oo, status = self.sm2pke_encrypt_packed_vartime(data, offs, k, Pb, mode, compressed)
        return [out[int(oo[i]):int(oo[i + 1])].tobytes() if status[i] == 1 else None for i in range(len(msgs))], status

    def sm2pke_decrypt_vartime(self, cts, d, mode="c1c3c2"):
        """DecryptingKey::decrypt over a list of ciphertexts (sm2/src/pke/decrypting.rs:174-222) -> plaintext bytes, or None
        where the reference returns Err"""
        data, offs = self._pack_messages(cts)
        out, pt_len, valid = self.sm2pke_decrypt_packed_vartime(data, offs, d, mode)
        return [out[int(offs[i]):int(offs[i]) + int(pt_len[i])].tobytes() if valid[i] else None for i in range(len(cts))]

    def sm2pke_encrypt(self, msgs, k, Pb, mode="c1c3c2", compressed: bool = True):
        self._sm2pke_ct("sm2pke_encrypt")
        return self.sm2pke_encrypt_vartime(msgs, k, Pb, mode, compressed)

    def sm2pke_decrypt(self, cts, d, mode="c1c3c2"):
        self._sm2pke_ct("sm2pke_decrypt")
        return self.sm2pke_decrypt_vartime(cts, d, mode)

    def sm2pke_encrypt_packed(self, data, offsets, k, Pb, mode="c1c3c2", compressed: bool = True):
        self._sm2pke_ct("sm2pke_encrypt_packed")
        return self.sm2pke_encrypt_packed_vartime(data, offsets, k, Pb, mode, compressed)

    def sm2pke_decrypt_packed(self, data, offsets, d, mode="c1c3c2"):
        self._sm2pke_ct("sm2pke_decrypt_packed")
        return self.sm2pke_decrypt_packed_vartime(data, offsets, d, mode)

    def sm2pke_encrypt_ptr(self, n, msgs, offsets, k32, Pb_xy, mode, compressed, out, status):
        """device-pointer mode (device_ptrs=True): every argument an integer CUDA address"""
        self._check(self.lib.ecg_sm2pke_encrypt_batch(self._ctx, n, _ptr(msgs), _ptr(offsets), _ptr(k32), _ptr(Pb_xy), SM2PKE_MODES[mode],
                                                      1 if compressed else 0, _ptr(out), _ptr(status)))

    def sm2pke_decrypt_ptr(self, n, cts, offsets, d32, mode, out, pt_len, valid):
        self._check(self.lib.ecg_sm2pke_decrypt_batch(self._ctx, n, _ptr(cts), _ptr(offsets), _ptr(d32), SM2PKE_MODES[mode], _ptr(out),
                                                      _ptr(pt_len), _ptr(valid)))

    def decompress_batch(self, curve, sec1_33):
        """AffinePoint::decompress over a batch of (1 + FB)-byte SEC1 compressed records -> (xy, inf, valid)"""
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(sec1_33).size // (fb + 1)
        sec1_33 = _u8(sec1_33, (fb + 1) * n, "sec1")
        out_xy = np.empty(2 * fb * n, np.uint8)
        out_inf = np.empty(n, np.uint8)
        valid = np.empty(n, np.uint8)
        self._check(self.lib.ecg_decompress_batch(self._ctx, c, n, _ptr(sec1_33), _ptr(out_xy), _ptr(out_inf), _ptr(valid)))
        return out_xy.reshape(n, 2 * fb), out_inf, valid

    @staticmethod
    def sec1_compress(xy, inf=None):
        """`GroupEncoding::to_bytes` / `to_sec1_point(true)` for a batch of affine outputs (primeorder/src/affine.rs:387-402):
        33-byte records, tag 02/03 by the parity of y then x; the identity is 33 zero bytes.  Pure byte shuffling on
        the host — the arithmetic (normalisation) already happened on the device."""
        xy = np.ascontiguousarray(xy, dtype=np.uint8).reshape(-1, 64)
        out = np.zeros((xy.shape[0], 33), np.uint8)
        out[:, 0] = 2 + (xy[:, 63] & 1)
        out[:, 1:] = xy[:, :32]
        if inf is not None:
            out[np.asarray(inf).reshape(-1) != 0] = 0
        return out

    def derive_public_keys_vartime(self, curve, secret_k, compressed=True):
        """Public-key derivation batch: `PublicKey::from_secret_scalar` = k * G, SEC1-encoded (SURVEY 8(f) rank 3;
        k256/src/schnorr/signing.rs:151 does the same for BIP340 keys).  Returns (records, inf).  VARIABLE TIME in the
        secret (table gathers by scalar digit) — see diffie_hellman_vartime; zero scalars are refused like NonZeroScalar."""
        n = np.asarray(secret_k).size // 32
        kk = _u8(secret_k, 32 * n, "secret_k").reshape(n, 32)
        if n and not kk.any(axis=1).all():
            raise ValueError("derive_public_keys_vartime: zero secret scalar (the reference takes a NonZeroScalar)")
        xy, inf = self.mul_by_generator(curve, secret_k)
        if compressed:
            return self.sec1_compress(xy, inf), inf
        out = np.zeros((xy.shape[0], 65), np.uint8)
        out[:, 0] = 4
        out[:, 1:] = xy
        out[inf != 0] = 0
        return out, inf

    def batch_normalize(self, curve, xyz):
        c = CURVE_IDS[curve]
        xyz = np.ascontiguousarray(xyz, dtype=np.uint8).reshape(-1)
        fb = FBYTES[c]
        n = xyz.size // (3 * fb)
        out_xy = np.empty(2 * fb * n, np.uint8)
        out_inf = np.empty(n, np.uint8)
        self._check(self.lib.ecg_batch_normalize(self._ctx, c, n, _ptr(xyz), _ptr(out_xy), _ptr(out_inf)))
        return out_xy.reshape(n, 2 * fb), out_inf

    def batch_normalize_hom(self, curve, xyz):
        """BatchNormalize for the reference's own homogeneous (X:Y:Z), x = X/Z (ecg_batch_normalize_hom)"""
        c = CURVE_IDS[curve]
        xyz = np.ascontiguousarray(xyz, dtype=np.uint8).reshape(-1)
        fb = FBYTES[c]
        n = xyz.size // (3 * fb)
        out_xy = np.empty(2 * fb * n, np.uint8)
        out_inf = np.empty(n, np.uint8)
        self._check(self.lib.ecg_batch_normalize_hom(self._ctx, c, n, _ptr(xyz), _ptr(out_xy), _ptr(out_inf)))
        return out_xy.reshape(n, 2 * fb), out_inf

    def field_sqrt(self, curve, a):
        """FieldElement::sqrt over a batch -> (roots n x FB, is_square)"""
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(a).size // fb
        a = _u8(a, fb * n, "a")
        out = np.empty(fb * n, np.uint8)
        ok = np.empty(n, np.uint8)
        self._check(self.lib.ecg_field_sqrt_batch(self._ctx, c, n, _ptr(a), _ptr(out), _ptr(ok)))
        return out.reshape(n, fb), ok

    def field_op(self, curve, op, a, b=None):
        c = CURVE_IDS[curve]
        fb = FBYTES[c]
        n = np.asarray(a).size // fb
        a = _u8(a, fb * n, "a")
        if b is not None:
            b = _u8(b, fb * n, "b")
        out = np.empty(fb * n, np.uint8)
        self._check(self.lib.ecg_field_op_batch(self._ctx, c, FOP[op] if isinstance(op, str) else op, n, _ptr(a), _ptr(b), _ptr(out)))
        return out.reshape(n, fb)

    # ---- raw-pointer API (device_ptrs=True): all arguments are integer CUDA device addresses ----
    def mul_batch_ptr(self, curve, n, k, P_xy, P_inf, out_xy, out_inf):
        self._check(self.lib.ecg_mul_batch(self._ctx, CURVE_IDS[curve], n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out_xy), _ptr(out_inf)))

    def mul_gen_batch_ptr(self, curve, n, k, out_xy, out_inf):
        self._check(self.lib.ecg_mul_gen_batch(self._ctx, CURVE_IDS[curve], n, _ptr(k), _ptr(out_xy), _ptr(out_inf)))

    def lincomb_partial_ptr(self, curve, n, k, P_xy, P_inf, out_xyz):
        self._check(self.lib.ecg_lincomb_partial(self._ctx, CURVE_IDS[curve], n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out_xyz)))

    def lincomb_ptr(self, curve, n, k, P_xy, P_inf, out_xy, out_inf):
        self._check(self.lib.ecg_lincomb(self._ctx, CURVE_IDS[curve], n, _ptr(k), _ptr(P_xy), _ptr(P_inf), _ptr(out_xy), _ptr(out_inf)))

    def point_sum_ptr(self, curve, m, xyz, out_xy, out_inf):
        """sum of m Jacobian points (m*96 bytes in device memory, e.g. an all_gather receive buffer) -> affine, on the device"""
        self._check(self.lib.ecg_point_sum(self._ctx, CURVE_IDS[curve], m, _ptr(xyz), _ptr(out_xy), _ptr(out_inf)))

    def schnorr_verify_ptr(self, n, pk_x, msg32, sig64, valid):
        self._check(self.lib.ecg_schnorr_verify_batch(self._ctx, n, _ptr(pk_x), _ptr(msg32), _ptr(sig64), _ptr(valid)))

    def timing_enable(self, on: bool = True):
        self._check(self.lib.ecg_timing_enable(self._ctx, 1 if on else 0))

    def timing_read(self):
        """(accumulated ms of the dominant kernel, number of calls) since timing_enable"""
        ms = ctypes.c_double(0)
        calls = ctypes.c_uint64(0)
        self._check(self.lib.ecg_timing_read(self._ctx, ctypes.byref(ms), ctypes.byref(calls)))
        return ms.value, int(calls.value)

    def microbench(self, which: int, iters: int = 2000):
        ops = ctypes.c_double(0)
        ms = ctypes.c_double(0)
        self._check(self.lib.ecg_microbench(self._ctx, which, iters, ctypes.byref(ops), ctypes.byref(ms)))
        return ops.value, ms.value
