"""SM2 public-key encryption and decryption (sm2/src/pke.rs, pke/encrypting.rs:166-230, pke/decrypting.rs:174-222) with the
SM3 KDF, in both ciphertext layouts (C1C3C2, C1C2C3).

Pinned to the GB/T 32905 SM3 vectors (and to hashlib's SM3 where it has one), to the reference's vectors
(sm2/tests/sm2pke.rs:10-21: CIPHER, and the OpenSSL-made ASN1_CIPHER restated as raw records in both layouts) and to
OpenSSL-made ciphertexts (oracle/make_sm2pke_golden.py), all in tests/golden/sm2_pke.json; the model's own ciphertexts
decrypt under the `openssl` command line where it is installed.  Compact C1 (tag 05) is decoded as primeorder's
`decompact` does (primeorder/src/affine.rs:64-73, 221-229); whether the reference accepts that tag at all is decided by the
`sec1` crate, which is not in the reference tree, so acceptance of tag 05 is unpinned.
CPU: the kernels on the host (tests/sim).  GPU: through the C ABI."""
import ctypes
import hashlib
import json
import os
import random
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import pyref
import sm2pke_ref

HERE = os.path.dirname(os.path.abspath(__file__))
C = pyref.CURVES["sm2"]
GOLD = json.load(open(os.path.join(HERE, "golden", "sm2_pke.json")))
REF = GOLD["reference"]
REF_D = int(REF["private_key"], 16)
OSSL_KEYS = [int(k, 16) for k in GOLD["openssl"]["keys"]]
OSSL = GOLD["openssl"]["vectors"]
# the plaintext lengths that cross the 32-byte KDF blocks and the 55 / 56-byte padding boundary of C3 = SM3(x2 || M || y2)
SWEEP = (0, 1, 2, 31, 32, 33, 55, 56, 57, 63, 64, 65, 119, 120, 121, 200)

_HAS_SM3 = "sm3" in hashlib.algorithms_available
# the model with hashlib's SM3 where it exists (pinned to sm2pke_ref.sm3 below), the pure-Python one elsewhere
SM3 = (lambda b: hashlib.new("sm3", b).digest()) if _HAS_SM3 else sm2pke_ref.sm3


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


def _pack(recs):
    offs = np.zeros(len(recs) + 1, np.uint64)
    offs[1:] = np.cumsum([len(r) for r in recs], dtype=np.uint64) if recs else []
    data = np.frombuffer(b"".join(recs) + b"\0", np.uint8).copy()
    return data, offs


def _msg(rng, L):
    return bytes(rng.getrandbits(8) for _ in range(L))


def _pub(d):
    return pyref.mul(C, d, pyref.G(C))


def _xy(P):
    return P[0].to_bytes(32, "big") + P[1].to_bytes(32, "big")


def model_encrypt_batch(Pbs, ks, msgs, mode, compressed):
    """the model over a batch, with the scalar multiplications in the C restatement (oracle/ecref_prime.c)"""
    import ecref
    n = len(ks)
    good = [0 < k < C.n and pyref.on_curve(C, P) and len(m) > 0 for k, P, m in zip(ks, Pbs, msgs)]
    Ks = np.frombuffer(b"".join((k if g else 1).to_bytes(32, "big") for k, g in zip(ks, good)), np.uint8).copy()
    PB = np.frombuffer(b"".join(_xy(P) if g else _xy(pyref.G(C)) for P, g in zip(Pbs, good)), np.uint8).copy()
    c1, _ = ecref.mul_gen_batch("sm2", Ks, nthreads=os.cpu_count() or 4)
    s, _ = ecref.mul_batch("sm2", Ks, PB, None, nthreads=os.cpu_count() or 4)
    c1, s = np.asarray(c1).reshape(n, 64), np.asarray(s).reshape(n, 64)
    out = []
    for i in range(n):
        if not good[i]:
            out.append((0, None))
            continue
        C1 = (int.from_bytes(c1[i, :32].tobytes(), "big"), int.from_bytes(c1[i, 32:].tobytes(), "big"))
        x2, y2 = int.from_bytes(s[i, :32].tobytes(), "big"), int.from_bytes(s[i, 32:].tobytes(), "big")
        out.append(sm2pke_ref.sm2pke_seal(C1, x2, y2, msgs[i], mode, compressed, SM3))
    return out


def model_decrypt_batch(ds, cts, mode):
    import ecref
    n = len(cts)
    parsed = [sm2pke_ref.sm2pke_parse(c, mode) if 0 < d < C.n else None for d, c in zip(ds, cts)]
    D = np.frombuffer(b"".join((d if p else 1).to_bytes(32, "big") for d, p in zip(ds, parsed)), np.uint8).copy()
    P = np.frombuffer(b"".join(_xy(p[0]) if p else _xy(pyref.G(C)) for p in parsed), np.uint8).copy()
    s, _ = ecref.mul_batch("sm2", D, P, None, nthreads=os.cpu_count() or 4)
    s = np.asarray(s).reshape(n, 64)
    return [None if p is None else sm2pke_ref.sm2pke_open(int.from_bytes(s[i, :32].tobytes(), "big"), int.from_bytes(s[i, 32:].tobytes(), "big"),
                                                       p[1], p[2], SM3) for i, p in enumerate(parsed)]


def expected_dec_out(cts, pts):
    """the decryption output buffer the ABI defines: plaintext at the start of each record's range, zeros elsewhere"""
    out = bytearray()
    for c, m in zip(cts, pts):
        out += (m or b"") + bytes(len(c) - len(m or b""))
    return bytes(out)


def expected_enc_out(res, msgs, compressed):
    ovh = 32 + (33 if compressed else 65)
    return b"".join(ct if st == 1 else bytes(len(m) + ovh) for (st, ct), m in zip(res, msgs))


def to_compact(ct):
    return b"\x05" + ct[1:33] + ct[33:] if ct[0] in (2, 3) else None


def k_with_small_y(rng):
    """an ephemeral scalar whose C1 = [k]G has y = min(y, p - y): its compact encoding decodes to C1 itself"""
    while True:
        k = rng.randrange(1, C.n)
        if _pub(k)[1] <= C.p - _pub(k)[1]:
            return k


# ---- model ------------------------------------------------------------------------------------------------------
def test_sm3_model_vectors():
    """GB/T 32905-2016 appendix A, and hashlib's SM3 (where the OpenSSL build has it) for lengths 0-300"""
    assert sm2pke_ref.sm3(b"abc").hex() == "66c7f0f462eeedd9d1f2d46bdc10e4e24167c4875cf2f7a2297da02b8f4ba8e0"
    assert sm2pke_ref.sm3(b"abcd" * 16).hex() == "debe9ff92275b8a138604889c18e5a4d6fdb70e5387e5765293dcba39c0c5732"
    if _HAS_SM3:
        rng = random.Random(5)
        for L in range(301):
            m = _msg(rng, L)
            assert sm2pke_ref.sm3(m) == hashlib.new("sm3", m).digest(), L


def test_model_decrypts_the_reference_vectors():
    M = REF["msg"].encode()
    assert sm2pke_ref.sm2pke_decrypt(REF_D, bytes.fromhex(REF["cipher_c1c3c2"]), 0) == M
    assert sm2pke_ref.sm2pke_decrypt(REF_D, bytes.fromhex(REF["asn1_as_c1c3c2"]), 0) == M
    assert sm2pke_ref.sm2pke_decrypt(REF_D, bytes.fromhex(REF["asn1_as_c1c2c3"]), 1) == M
    assert sm2pke_ref.sm2pke_decrypt(REF_D, bytes.fromhex(REF["cipher_c1c3c2"]), 1) is None
    assert sm2pke_ref.sm2pke_decrypt(REF_D + 1, bytes.fromhex(REF["cipher_c1c3c2"]), 0) is None


def test_model_decrypts_the_openssl_fixtures():
    assert len(OSSL) >= 40 and {v["len"] for v in OSSL} >= {1, 31, 32, 33, 55, 56, 63, 64, 65, 119, 120, 1000, 4096}
    for v in OSSL:
        d, M = OSSL_KEYS[v["key"]], bytes.fromhex(v["msg"])
        assert sm2pke_ref.sm2pke_decrypt(d, bytes.fromhex(v["c1c3c2"]), 0) == M
        assert sm2pke_ref.sm2pke_decrypt(d, bytes.fromhex(v["c1c2c3"]), 1) == M


def _der_int(v):
    b = v.to_bytes(33, "big").lstrip(b"\0")
    b = b"\0" + b if not b or b[0] & 0x80 else b
    return b"\x02" + bytes([len(b)]) + b


def _der(tag, body):
    n = len(body)
    return bytes([tag]) + (bytes([n]) if n < 0x80 else bytes([0x82, n >> 8, n & 0xFF])) + body


@pytest.mark.skipif(shutil.which("openssl") is None, reason="no openssl command line")
def test_model_ciphertexts_decrypt_under_openssl():
    """the model's C1C3C2 ciphertexts, in the GM/T 0009 DER form `openssl pkeyutl -decrypt` reads"""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "oracle"))
    from make_sm2pke_golden import key_pem
    rng = random.Random(11)
    d = OSSL_KEYS[1]
    with tempfile.TemporaryDirectory() as td:
        kp = os.path.join(td, "k.pem")
        open(kp, "w").write(key_pem(d))
        for L in (1, 32, 56, 65, 300):
            M = _msg(rng, L)
            st, ct = sm2pke_ref.sm2pke_encrypt(_pub(d), rng.randrange(1, C.n), M, 0, False)
            assert st == 1
            der = _der(0x30, _der_int(int.from_bytes(ct[1:33], "big")) + _der_int(int.from_bytes(ct[33:65], "big")) +
                       _der(0x04, ct[65:97]) + _der(0x04, ct[97:]))
            cp = os.path.join(td, "c")
            open(cp, "wb").write(der)
            r = subprocess.run(["openssl", "pkeyutl", "-decrypt", "-inkey", kp, "-in", cp], capture_output=True)
            assert r.returncode == 0 and r.stdout == M, (L, r.stderr)


# ---- kernels on the host --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sim():
    import __graft_entry__ as ge
    ge.build()
    return ctypes.CDLL(os.path.join(HERE, "sim", "libecgsim_sm2pke.so"))


def test_device_sm3_on_host(sim):
    rng = random.Random(1)
    out = np.zeros(32, np.uint8)
    for L in range(301):
        m = np.frombuffer(_msg(rng, L) + b"\0", np.uint8).copy()
        sim.simk_sm3(_p(m), ctypes.c_size_t(L), _p(out))
        assert out.tobytes() == sm2pke_ref.sm3(m[:L].tobytes()), L


def sim_decrypt(sim, cts, ds, mode):
    data, offs = _pack(cts)
    D = np.frombuffer(b"".join((d % (1 << 256)).to_bytes(32, "big") for d in ds), np.uint8).copy()
    out = np.full(max(int(offs[-1]), 1), 0xAB, np.uint8)
    pt_len = np.full(len(cts), 77, np.uint64)
    valid = np.full(len(cts), 9, np.uint8)
    assert sim.simk_sm2pke_decrypt(ctypes.c_size_t(len(cts)), _p(data), _p(offs), _p(D), mode, _p(out), _p(pt_len), _p(valid)) == 0
    return out[:int(offs[-1])].tobytes(), pt_len, valid


def sim_encrypt(sim, msgs, ks, Pbs, mode, compressed, table=None):
    data, offs = _pack(msgs)
    K = np.frombuffer(b"".join((k % (1 << 256)).to_bytes(32, "big") for k in ks), np.uint8).copy()
    PB = np.frombuffer(b"".join(_xy(P) for P in Pbs), np.uint8).copy()
    ovh = 32 + (33 if compressed else 65)
    out = np.full(int(offs[-1]) + ovh * len(msgs) + 1, 0xAB, np.uint8)
    status = np.full(len(msgs), 9, np.uint8)
    rc = sim.simk_sm2pke_encrypt(ctypes.c_size_t(len(msgs)), _p(data), _p(offs), _p(K), _p(PB), mode, 1 if compressed else 0,
                                 None if table is None else _p(table), _p(out), _p(status))
    assert rc == 0
    return out[:-1].tobytes(), status


def _check_dec(sim, cts, ds, mode):
    out, pt_len, valid = sim_decrypt(sim, cts, ds, mode)
    exp = [sm2pke_ref.sm2pke_decrypt(d, c, mode) for d, c in zip(ds, cts)]
    assert [bool(v) for v in valid] == [m is not None for m in exp]
    assert [int(x) for x in pt_len] == [len(m) if m is not None else 0 for m in exp]
    assert out == expected_dec_out(cts, exp)
    return exp


def test_decrypt_kernels_on_host_vectors(sim):
    M = REF["msg"].encode()
    cts = [bytes.fromhex(REF["cipher_c1c3c2"]), bytes.fromhex(REF["asn1_as_c1c3c2"])]
    assert _check_dec(sim, cts, [REF_D] * 2, 0) == [M, M]
    assert _check_dec(sim, [bytes.fromhex(REF["asn1_as_c1c2c3"])], [REF_D], 1) == [M]
    for mode, key in ((0, "c1c3c2"), (1, "c1c2c3")):
        vs = [v for v in OSSL if v["len"] <= 120]
        exp = _check_dec(sim, [bytes.fromhex(v[key]) for v in vs], [OSSL_KEYS[v["key"]] for v in vs], mode)
        assert exp == [bytes.fromhex(v["msg"]) for v in vs]


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("form", ["compressed", "uncompressed", "compact"])
def test_decrypt_kernels_on_host_sweep(sim, mode, form):
    rng = random.Random(100 + mode * 3 + len(form))
    cts, ds = [], []
    for L in SWEEP[1:]:
        d = rng.randrange(1, C.n)
        k = k_with_small_y(rng) if form == "compact" else rng.randrange(1, C.n)
        st, ct = sm2pke_ref.sm2pke_encrypt(_pub(d), k, _msg(rng, L), mode, form != "uncompressed")
        assert st == 1
        cts.append(to_compact(ct) if form == "compact" else ct)
        ds.append(d)
    exp = _check_dec(sim, cts, ds, mode)
    assert all(m is not None for m in exp)


def test_decrypt_rejections_on_host(sim):
    """each corruption gives valid = 0 and an all-zero record range"""
    rng = random.Random(7)
    d = rng.randrange(1, C.n)
    M = _msg(rng, 70)
    _, cu = sm2pke_ref.sm2pke_encrypt(_pub(d), rng.randrange(1, C.n), M, 0, False)
    _, cc = sm2pke_ref.sm2pke_encrypt(_pub(d), rng.randrange(1, C.n), M, 0, True)
    bad, keys = [], []

    def add(ct, key=d):
        bad.append(ct)
        keys.append(key)

    for ct in (cu, cc):
        for pos in (1, 20, len(ct) - 70 - 32, len(ct) - 70 - 1, len(ct) - 70, len(ct) - 1):   # C1, C3, C2
            b = bytearray(ct)
            b[pos] ^= 0x10
            add(bytes(b))
        c1len = 65 if ct is cu else 33
        add(ct[:c1len + 31])                              # truncation below C1 + 32
        add(ct[:c1len])
        for tag in (0x00, 0x01, 0x06, 0x07):
            add(bytes([tag]) + ct[1:])
    add(b"")
    add(b"\x00" * 40)                                     # the identity: [h]C1 = O
    add(b"\x04" + C.p.to_bytes(32, "big") + cu[33:])      # x >= p
    x = next(x for x in range(2, 1000) if pow((x ** 3 - 3 * x + C.b) % C.p, (C.p - 1) // 2, C.p) != 1)
    add(b"\x02" + x.to_bytes(32, "big") + cc[33:])        # compressed x without a square root
    add(cu, 0)
    add(cu, C.n)
    add(cu, C.n + 5)
    out, pt_len, valid = sim_decrypt(sim, bad, keys, 0)
    assert not valid.any() and not pt_len.any() and not any(out), [i for i, v in enumerate(valid) if v]
    out, pt_len, valid = sim_decrypt(sim, [cu, cc], [d, d], 1)   # the wrong mode
    assert not valid.any() and not any(out)
    out, pt_len, valid = sim_decrypt(sim, [cu, cc], [d, d], 0)
    assert valid.all() and out == M + bytes(len(cu) - 70) + M + bytes(len(cc) - 70)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("compressed", [True, False])
def test_encrypt_kernels_on_host_sweep(sim, mode, compressed):
    """[k]G through the variable-base routine (the ECG_FLAG_CONSTTIME path)"""
    rng = random.Random(200 + 2 * mode + compressed)
    msgs = [_msg(rng, L) for L in SWEEP[1:]]
    ks = [rng.randrange(1, C.n) for _ in msgs]
    Pbs = [_pub(rng.randrange(1, C.n)) for _ in msgs]
    out, status = sim_encrypt(sim, msgs, ks, Pbs, mode, compressed)
    exp = [sm2pke_ref.sm2pke_encrypt(P, k, m, mode, compressed) for P, k, m in zip(Pbs, ks, msgs)]
    assert [int(s) for s in status] == [e[0] for e in exp] == [1] * len(msgs)
    assert out == expected_enc_out(exp, msgs, compressed)


def test_encrypt_kernels_on_host_fixed_base_table(sim):
    """[k]G by the fixed-base table (the default path), and the refusals: k = 0, k >= n, Pb off the curve, empty M"""
    from test_curves_ext import ext_fb_table
    table = ext_fb_table(sim, pyref.CURVE_IDS["sm2"])
    rng = random.Random(300)
    msgs = [_msg(rng, L) for L in (1, 33, 56, 64, 65)] + [b"abc", b"abc", b"abc", b""]
    ks = [rng.randrange(1, C.n) for _ in range(5)] + [0, C.n, 5, 7]
    P = _pub(rng.randrange(1, C.n))
    Pbs = [P] * 7 + [(P[0], (P[1] + 1) % C.p), P]
    for mode in (0, 1):
        out, status = sim_encrypt(sim, msgs, ks, Pbs, mode, True, table)
        exp = [sm2pke_ref.sm2pke_encrypt(Pb, k, m, mode, True) for Pb, k, m in zip(Pbs, ks, msgs)]
        assert [int(s) for s in status] == [e[0] for e in exp] == [1] * 5 + [0] * 4
        assert out == expected_enc_out(exp, msgs, True)


# ---- on the GPU -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng():
    import ecgpu
    e = ecgpu.Engine()
    yield e
    e.close()


@pytest.mark.gpu
def test_gpu_vectors_and_fixtures(eng):
    M = REF["msg"].encode()
    assert eng.sm2pke_decrypt_vartime([bytes.fromhex(REF["cipher_c1c3c2"]), bytes.fromhex(REF["asn1_as_c1c3c2"])], REF_D.to_bytes(32, "big")) == [M, M]
    assert eng.sm2pke_decrypt_vartime([bytes.fromhex(REF["asn1_as_c1c2c3"])], REF_D.to_bytes(32, "big"), "c1c2c3") == [M]
    assert eng.sm2pke_decrypt_vartime([bytes.fromhex(REF["cipher_c1c3c2"])], REF_D.to_bytes(32, "big"), "c1c2c3") == [None]
    D = np.frombuffer(b"".join(OSSL_KEYS[v["key"]].to_bytes(32, "big") for v in OSSL), np.uint8)
    for mode in ("c1c3c2", "c1c2c3"):
        got = eng.sm2pke_decrypt_vartime([bytes.fromhex(v[mode]) for v in OSSL], D, mode)
        assert got == [bytes.fromhex(v["msg"]) for v in OSSL]


def _random_batch(seed, n, lmax, keys=None):
    rng = random.Random(seed)
    msgs = [_msg(rng, rng.randrange(0, lmax + 1)) for _ in range(n)]
    ds = keys or [rng.randrange(1, C.n) for _ in range(n)]
    ks = [rng.randrange(1, C.n) for _ in range(n)]
    return rng, msgs, ds, ks


@pytest.mark.gpu
def test_gpu_random_4096_against_the_model(eng):
    """4096 records, lengths uniform in 0-1024, one key pair per record: GPU encryption == the model byte for byte (both
    layouts, both C1 forms), GPU decryption of those plus corrupted ones == the model"""
    import ecref
    rng, msgs, ds, ks = _random_batch(41, 4096, 1024)
    Dk = np.frombuffer(b"".join(d.to_bytes(32, "big") for d in ds), np.uint8).copy()
    pub, _ = ecref.mul_gen_batch("sm2", Dk, nthreads=os.cpu_count() or 4)
    pub = np.asarray(pub).reshape(-1, 64)
    Pbs = [(int.from_bytes(r[:32].tobytes(), "big"), int.from_bytes(r[32:].tobytes(), "big")) for r in pub]
    K = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8).copy()
    for mode, compressed in ((0, True), (1, False)):
        cts, status = eng.sm2pke_encrypt_vartime(msgs, K, pub, mode, compressed)
        exp = model_encrypt_batch(Pbs, ks, msgs, mode, compressed)
        assert [int(s) for s in status] == [e[0] for e in exp]
        assert sum(status == 0) == sum(len(m) == 0 for m in msgs)
        bad = [i for i, (c, e) in enumerate(zip(cts, exp)) if c != e[1]]
        assert not bad, f"ciphertext differs from the model at {bad[:8]}"
        # decryption: the valid ones, every 7th corrupted, every 11th under the wrong key
        dcts = [c if c is not None else b"\x04" for c in cts]
        dds = list(ds)
        for i in range(0, 4096, 7):
            b = bytearray(dcts[i])
            b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
            dcts[i] = bytes(b)
        for i in range(3, 4096, 11):
            dds[i] = (ds[i] % (C.n - 1)) + 1
        D = np.frombuffer(b"".join(d.to_bytes(32, "big") for d in dds), np.uint8).copy()
        data, offs = _pack(dcts)
        out, pt_len, valid = eng.sm2pke_decrypt_packed_vartime(data, offs, D, mode)
        pts = model_decrypt_batch(dds, dcts, mode)
        assert [bool(v) for v in valid] == [m is not None for m in pts]
        assert out.tobytes() == expected_dec_out(dcts, pts)
        assert sum(m is not None for m in pts) > 3000


@pytest.mark.gpu
def test_gpu_seeded_encrypt_equals_model_and_decrypt_inverts(eng):
    rng, msgs, _, ks = _random_batch(5, 300, 300)
    d = rng.randrange(1, C.n)
    Pb = _pub(d)
    for mode in ("c1c3c2", "c1c2c3"):
        for compressed in (True, False):
            cts, status = eng.sm2pke_encrypt_vartime(msgs, np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8), _xy(Pb),
                                                     mode, compressed)
            for i in (0, 1, 17, 299):
                assert (int(status[i]), cts[i]) == sm2pke_ref.sm2pke_encrypt(Pb, ks[i], msgs[i], 0 if mode == "c1c3c2" else 1, compressed)
            back = eng.sm2pke_decrypt_vartime([c or b"" for c in cts], d.to_bytes(32, "big"), mode)
            assert back == [m if len(m) else None for m in msgs]


@pytest.mark.gpu
def test_gpu_consttime_and_zeroize_ctx_agree():
    import ecgpu
    rng, msgs, ds, ks = _random_batch(9, 1000, 200)
    K = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8).copy()
    Pb = _xy(_pub(ds[0]))
    res = []
    for kw in ({}, {"consttime": True}, {"zeroize": True}, {"consttime": True, "zeroize": True}):
        e = ecgpu.Engine(**kw)
        enc = e.sm2pke_encrypt if kw.get("consttime") else e.sm2pke_encrypt_vartime
        dec = e.sm2pke_decrypt if kw.get("consttime") else e.sm2pke_decrypt_vartime
        cts, status = enc(msgs, K, Pb, "c1c2c3", False)
        pts = dec([c or b"" for c in cts], ds[0].to_bytes(32, "big"), "c1c2c3")
        res.append((cts, status.tolist(), pts))
        if not kw.get("consttime"):
            with pytest.raises(ValueError):
                e.sm2pke_decrypt([b""], ds[0].to_bytes(32, "big"))
        e.close()
    assert all(r == res[0] for r in res[1:])
    assert res[0][2] == [m if len(m) else None for m in msgs]


@pytest.mark.gpu
def test_gpu_device_pointers_with_torch():
    import torch

    import ecgpu
    rng, msgs, ds, ks = _random_batch(13, 500, 300)
    d = ds[0]
    Pb = _pub(d)
    ref = model_encrypt_batch([Pb] * 500, ks, msgs, 0, True)
    host = ecgpu.Engine()
    e = ecgpu.Engine(device_ptrs=True)
    dev = torch.device("cuda:0")
    data, offs = _pack(msgs)
    t_data = torch.from_numpy(data).to(dev)
    t_offs = torch.from_numpy(offs.view(np.int64)).to(dev)
    t_k = torch.from_numpy(np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8).copy()).to(dev)
    t_pb = torch.from_numpy(np.frombuffer(_xy(Pb) * 500, np.uint8).copy()).to(dev)
    total = int(offs[-1]) + 500 * 65
    t_out = torch.full((total,), 0xAB, dtype=torch.uint8, device=dev)
    t_st = torch.zeros(500, dtype=torch.uint8, device=dev)
    e.sm2pke_encrypt_ptr(500, t_data.data_ptr(), t_offs.data_ptr(), t_k.data_ptr(), t_pb.data_ptr(), 0, True, t_out.data_ptr(), t_st.data_ptr())
    torch.cuda.synchronize()
    assert t_out.cpu().numpy().tobytes() == expected_enc_out(ref, msgs, True)
    assert t_st.cpu().numpy().tolist() == [r[0] for r in ref]
    # decrypt the records back in place on the device
    o_offs = (offs - offs[0]) + np.arange(501, dtype=np.uint64) * np.uint64(65)
    t_ooffs = torch.from_numpy(o_offs.view(np.int64)).to(dev)
    t_d = torch.from_numpy(np.frombuffer(d.to_bytes(32, "big") * 500, np.uint8).copy()).to(dev)
    t_pt = torch.full((total,), 0xAB, dtype=torch.uint8, device=dev)
    t_len = torch.zeros(500, dtype=torch.int64, device=dev)
    t_ok = torch.zeros(500, dtype=torch.uint8, device=dev)
    e.sm2pke_decrypt_ptr(500, t_out.data_ptr(), t_ooffs.data_ptr(), t_d.data_ptr(), 0, t_pt.data_ptr(), t_len.data_ptr(), t_ok.data_ptr())
    torch.cuda.synchronize()
    cts = [r[1] or bytes(len(m) + 65) for r, m in zip(ref, msgs)]
    pts = [m if len(m) else None for m in msgs]
    assert t_ok.cpu().numpy().tolist() == [1 if p else 0 for p in pts]
    assert t_pt.cpu().numpy().tobytes() == expected_dec_out(cts, pts)
    # host mode on the same records agrees
    out, pt_len, valid = host.sm2pke_decrypt_packed_vartime(t_out.cpu().numpy(), o_offs, d.to_bytes(32, "big"))
    assert out.tobytes() == t_pt.cpu().numpy().tobytes()
    e.close()
    host.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 127, 129, 1000])
def test_gpu_ragged_sizes(eng, n):
    rng, msgs, ds, ks = _random_batch(1000 + n, n, 90)
    Pb = _pub(ds[0]) if n else pyref.G(C)
    K = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8).copy() if n else np.zeros(0, np.uint8)
    cts, status = eng.sm2pke_encrypt_vartime(msgs, K, _xy(Pb))
    assert len(cts) == n and status.size == n
    if n == 0:
        assert eng.sm2pke_decrypt_vartime([], bytes(32)) == []
        return
    assert cts == [e[1] for e in model_encrypt_batch([Pb] * n, ks, msgs, 0, True)]
    assert eng.sm2pke_decrypt_vartime([c or b"" for c in cts], ds[0].to_bytes(32, "big")) == [m if m else None for m in msgs]


@pytest.mark.gpu
def test_gpu_argument_errors(eng):
    import ecgpu
    lib = eng.lib
    ctx = eng._ctx
    data = np.zeros(200, np.uint8)
    offs = np.array([0, 100, 200], np.uint64)
    k = np.frombuffer((5).to_bytes(32, "big") * 2, np.uint8).copy()
    pb = np.frombuffer(_xy(pyref.G(C)) * 2, np.uint8).copy()
    out = np.zeros(400, np.uint8)
    st = np.zeros(2, np.uint8)
    ln = np.zeros(2, np.uint64)
    E = ecgpu.ECG_EINVAL

    def enc(n=2, d=data, o=offs, kk=k, p=pb, mode=0, ou=out, s=st):
        return lib.ecg_sm2pke_encrypt_batch(ctx, n, _ptr(d), _ptr(o), _ptr(kk), _ptr(p), mode, 1, _ptr(ou), _ptr(s))

    def dec(n=2, d=data, o=offs, kk=k, mode=0, ou=out, lp=ln, s=st):
        return lib.ecg_sm2pke_decrypt_batch(ctx, n, _ptr(d), _ptr(o), _ptr(kk), mode, _ptr(ou), _ptr(lp), _ptr(s))

    assert enc() == ecgpu.ECG_OK and dec() == ecgpu.ECG_OK
    assert lib.ecg_sm2pke_encrypt_batch(None, 2, _ptr(data), _ptr(offs), _ptr(k), _ptr(pb), 0, 1, _ptr(out), _ptr(st)) == E
    for bad in ({"o": None}, {"kk": None}, {"p": None}, {"ou": None}, {"s": None}, {"d": None}, {"mode": 2}, {"mode": -1},
                {"o": np.array([0, 150, 100], np.uint64)}):
        assert enc(**bad) == E, bad
    for bad in ({"o": None}, {"kk": None}, {"ou": None}, {"lp": None}, {"s": None}, {"d": None}, {"mode": 5},
                {"o": np.array([0, 150, 100], np.uint64)}):
        assert dec(**bad) == E, bad
    assert enc(n=0, d=None, o=None, kk=None, p=None, ou=None, s=None) == ecgpu.ECG_OK
    assert dec(n=0, d=None, o=None, kk=None, ou=None, lp=None, s=None) == ecgpu.ECG_OK
    # device-pointer mode: misaligned offsets / keys
    import torch
    e = ecgpu.Engine(device_ptrs=True)
    dev = torch.device("cuda:0")
    buf = torch.zeros(4096, dtype=torch.uint8, device=dev)
    base = buf.data_ptr()
    t_offs = torch.tensor([0, 0, 0, 0], dtype=torch.int64, device=dev)
    args = dict(n=2, msgs=base, offsets=t_offs.data_ptr(), k32=base + 1024, Pb_xy=base + 2048, out=base + 3072, status=base + 4000)
    for key, delta in (("offsets", 4), ("k32", 1), ("Pb_xy", 2)):
        a = dict(args)
        a[key] += delta
        assert e.lib.ecg_sm2pke_encrypt_batch(e._ctx, a["n"], _ptr(a["msgs"]), _ptr(a["offsets"]), _ptr(a["k32"]), _ptr(a["Pb_xy"]), 0, 1,
                                              _ptr(a["out"]), _ptr(a["status"])) == E, key
    assert e.lib.ecg_sm2pke_decrypt_batch(e._ctx, 2, _ptr(base), _ptr(t_offs.data_ptr()), _ptr(base + 1024), 0, _ptr(base + 3072),
                                          _ptr(base + 2052), _ptr(base + 4000)) == E    # pt_len not 8-byte aligned
    e.close()


def _ptr(a):
    if a is None:
        return ctypes.c_void_p(0)
    if isinstance(a, np.ndarray):
        return ctypes.c_void_p(a.ctypes.data)
    return ctypes.c_void_p(int(a))


CPP = r"""
#include <cstdio>
#include "ecgpu.hpp"
int main() {
  try {
    ecgpu::Engine eng(ECG_SM2);
    ecgpu::Scalar d{}, k1{}, k2{};
    d[31] = 7; k1[31] = 11; k2[31] = 13;
    ecgpu::AffinePoint pb = eng.mul_by_generator({d})[0];
    std::vector<uint8_t> st;
    auto cts = eng.sm2pke_encrypt(pb, {k1, k2}, {"hello", std::string(100, 'x')}, 1, false, &st);
    if (st.size() != 2 || st[0] != 1 || st[1] != 1 || cts[0].size() != 5 + 97 || cts[1].size() != 100 + 97) return 4;
    std::vector<bool> ok;
    auto pts = eng.sm2pke_decrypt(d, cts, 1, &ok);
    if (!ok[0] || !ok[1] || std::string(pts[0].begin(), pts[0].end()) != "hello" || pts[1].size() != 100) return 5;
    auto none = eng.sm2pke_decrypt(d, cts, 0, &ok);
    if (ok[0] || ok[1] || !none[0].empty()) return 6;
    for (auto b : cts[0]) printf("%02x", b);
    printf("\ncpp sm2pke ok\n");
  } catch (const std::exception& e) {
    fprintf(stderr, "%s\n", e.what());
    return 3;
  }
  return 0;
}
"""


@pytest.mark.gpu
def test_gpu_cpp_mirror():
    from test_host_cpp import _build_and_run
    rc, out = _build_and_run(CPP)
    assert rc == 0 and "cpp sm2pke ok" in out, out
    ct = bytes.fromhex(out.split()[0])
    assert (1, ct) == sm2pke_ref.sm2pke_encrypt(_pub(7), 11, b"hello", 1, False)
