"""SM3 and SM2 public-key encryption, pure Python: the model the device entries ecg_sm2pke_{encrypt,decrypt}_batch are
checked against.

TEST INFRASTRUCTURE ONLY, like pyref.py (whose curve arithmetic it uses): nothing in the product path imports it.
Each function restates the reference step by step (sm2/src/pke.rs, pke/encrypting.rs:166-230, pke/decrypting.rs:174-222);
the SM3 here is pinned to the GB/T 32905 vectors and, where hashlib has SM3, to hashlib (tests/test_sm2pke.py).
"""
from __future__ import annotations

from pyref import CURVES, G, mul, on_curve
# ---- SM3 (GB/T 32905-2016), pure Python: the digest of SM2 public-key encryption --------------------------------------
# hashlib has SM3 only where its OpenSSL build provides it; this model does not depend on that.
_SM3_IV = (0x7380166F, 0x4914B2B9, 0x172442D7, 0xDA8A0600, 0xA96F30BC, 0x163138AA, 0xE38DEE4D, 0xB0FB0E4E)


def _rotl32(x: int, n: int) -> int:
    n %= 32
    return ((x << n) | (x >> (32 - n))) & 0xFFFFFFFF


def _sm3_compress(v, block: bytes):
    p0 = lambda x: x ^ _rotl32(x, 9) ^ _rotl32(x, 17)    # noqa: E731
    p1 = lambda x: x ^ _rotl32(x, 15) ^ _rotl32(x, 23)   # noqa: E731
    w = [int.from_bytes(block[4 * i:4 * i + 4], "big") for i in range(16)]
    for j in range(16, 68):
        w.append(p1(w[j - 16] ^ w[j - 9] ^ _rotl32(w[j - 3], 15)) ^ _rotl32(w[j - 13], 7) ^ w[j - 6])
    a, b, c, d, e, f, g, h = v
    for j in range(64):
        tj = 0x79CC4519 if j < 16 else 0x7A879D8A
        ss1 = _rotl32((_rotl32(a, 12) + e + _rotl32(tj, j)) & 0xFFFFFFFF, 7)
        ss2 = ss1 ^ _rotl32(a, 12)
        ff = (a ^ b ^ c) if j < 16 else ((a & b) | (a & c) | (b & c))
        gg = (e ^ f ^ g) if j < 16 else ((e & f) | (~e & g))
        tt1 = (ff + d + ss2 + (w[j] ^ w[j + 4])) & 0xFFFFFFFF
        tt2 = (gg + h + ss1 + w[j]) & 0xFFFFFFFF
        a, b, c, d = tt1, a, _rotl32(b, 9), c
        e, f, g, h = p0(tt2), e, _rotl32(f, 19), g
    return tuple(x ^ y for x, y in zip(v, (a, b, c, d, e, f, g, h)))


def sm3(msg: bytes) -> bytes:
    """SM3 digest: SHA-256-style padding (0x80, zeros, 64-bit big-endian bit length), 64-byte blocks"""
    m = bytes(msg) + b"\x80" + bytes((55 - len(msg)) % 64) + (8 * len(msg)).to_bytes(8, "big")
    v = _SM3_IV
    for i in range(0, len(m), 64):
        v = _sm3_compress(v, m[i:i + 64])
    return b"".join(x.to_bytes(4, "big") for x in v)


# ---- SM2 public-key encryption (sm2/src/pke.rs, pke/encrypting.rs:166-230, pke/decrypting.rs:174-222), digest SM3 ----
SM2PKE_C1C3C2, SM2PKE_C1C2C3 = 0, 1   # pke.rs Mode; C1C3C2 is the reference's default


def sm2pke_kdf(x2: int, y2: int, klen: int, digest=sm3) -> bytes:
    """t = KDF(x2 || y2, klen): SM3(x2 || y2 || BE32(j)) for j = 1, 2, ..., truncated to klen bytes (pke.rs:349-381; the
    counter is `i32::try_from(index + 1)`, so klen < 2^31 * 32).  `digest`: any function equal to sm3 (a faster one)."""
    z = x2.to_bytes(32, "big") + y2.to_bytes(32, "big")
    return b"".join(digest(z + j.to_bytes(4, "big")) for j in range(1, (klen + 31) // 32 + 1))[:klen]


def sm2pke_c1_decode(c1: bytes):
    """FromSec1Point for sm2 (primeorder/src/affine.rs:204-229): 02/03 decompress by parity, 05 compact (decompress with
    even y, then y = min(y, p - y): to_compact, :64-73), 04 from_coordinates, 00 the identity -> point | None (invalid)"""
    c = CURVES["sm2"]
    tag = c1[0]
    if tag == 0:
        return "identity"
    x = int.from_bytes(c1[1:33], "big")
    if x >= c.p:
        return None
    if tag == 4:
        y = int.from_bytes(c1[33:65], "big")
        return (x, y) if on_curve(c, (x, y)) else None
    rhs = (x * x * x + c.a * x + c.b) % c.p
    y = pow(rhs, (c.p + 1) // 4, c.p)   # p = 3 (mod 4)
    if y * y % c.p != rhs:
        return None
    if (y & 1) != (tag == 3):
        y = c.p - y
    if tag == 5:
        y = min(y, c.p - y)
    return (x, y)


def sm2pke_seal(C1, x2: int, y2: int, M: bytes, mode: int = SM2PKE_C1C3C2, compressed: bool = True, digest=sm3):
    """A5-A7 and the layout, given C1 = [k]G and (x2, y2) = [k]Pb -> (status, ciphertext | None)"""
    t = sm2pke_kdf(x2, y2, len(M), digest)        # A5
    if not any(t):                                # encrypting.rs:202-205 (never true for an empty M: refused before)
        return 2, None
    C2 = (int.from_bytes(M, "big") ^ int.from_bytes(t, "big")).to_bytes(len(M), "big")   # A6
    C3 = digest(x2.to_bytes(32, "big") + M + y2.to_bytes(32, "big"))   # A7
    c1 = (bytes([2 | (C1[1] & 1)]) + C1[0].to_bytes(32, "big")) if compressed else (b"\x04" + C1[0].to_bytes(32, "big") + C1[1].to_bytes(32, "big"))
    return 1, c1 + (C3 + C2 if mode == SM2PKE_C1C3C2 else C2 + C3)   # Cipher::to_slice, pke.rs:181-213


def sm2pke_encrypt(Pb, k: int, M: bytes, mode: int = SM2PKE_C1C3C2, compressed: bool = True):
    """one pass of `encrypt` (encrypting.rs:166-230) with the caller's k -> (status, ciphertext | None):
    status 1 = ok; 0 = refused (k not in [1, n-1], Pb not on the curve, empty M: the reference's retry loop would never end,
    its all-zero test over zero bytes being false); 2 = t all zero (the reference draws another k)."""
    c = CURVES["sm2"]
    if not (0 < k < c.n) or Pb is None or not on_curve(c, Pb) or len(M) == 0:
        return 0, None
    C1 = mul(c, k, G(c))                          # A2: C1 = [k]G
    x2, y2 = mul(c, k, Pb)                        # A3, A4: [h]Pb != O (h = Scalar::S = 1 for sm2), (x2, y2) = [k]Pb
    return sm2pke_seal(C1, x2, y2, M, mode, compressed)


def sm2pke_parse(C: bytes, mode: int = SM2PKE_C1C3C2):
    """Cipher::from_slice (pke.rs:122-160) -> (C1, C2, C3) | None"""
    if len(C) == 0:
        return None
    c1len = {0: 1, 2: 33, 3: 33, 5: 33, 4: 65}.get(C[0])
    if c1len is None or len(C) < c1len + 32:
        return None
    P = sm2pke_c1_decode(C[:c1len])
    if P is None or P == "identity":              # [h]C1 = O is refused
        return None
    rest = C[c1len:]
    C3, C2 = (rest[:32], rest[32:]) if mode == SM2PKE_C1C3C2 else (rest[-32:], rest[:-32])
    return P, C2, C3


def sm2pke_open(x2: int, y2: int, C2: bytes, C3: bytes, digest=sm3):
    """B4-B6 given (x2, y2) = [d]C1 -> plaintext | None"""
    M = (int.from_bytes(C2, "big") ^ int.from_bytes(sm2pke_kdf(x2, y2, len(C2), digest), "big")).to_bytes(len(C2), "big")   # B4, B5
    # (an all-zero t is not refused on decryption)
    u = digest(x2.to_bytes(32, "big") + M + y2.to_bytes(32, "big"))             # B6
    return M if u == C3 else None


def sm2pke_decrypt(d: int, C: bytes, mode: int = SM2PKE_C1C3C2):
    """DecryptingKey::decrypt (Cipher::from_slice, then decrypting.rs:174-222) -> plaintext | None"""
    c = CURVES["sm2"]
    parsed = sm2pke_parse(C, mode)
    if not (0 < d < c.n) or parsed is None:
        return None
    P, C2, C3 = parsed
    x2, y2 = mul(c, d, P)                         # B3
    return sm2pke_open(x2, y2, C2, C3)
