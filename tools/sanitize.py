"""Small invocation of every C-ABI entry point, meant to be run under compute-sanitizer on the GPU box:
    compute-sanitizer --tool memcheck  --error-exitcode 9 python tools/sanitize.py
    compute-sanitizer --tool racecheck --error-exitcode 9 python tools/sanitize.py
    compute-sanitizer --tool initcheck --error-exitcode 9 python tools/sanitize.py
Sizes are tiny (the tools slow kernels 10-100x); results are still checked against the oracle port."""
import os, random, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "elliptic-curves_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import ecgpu, pyref, ecref, sm2pke_ref
from helpers import pack_scalars, pack_points, unpack_points

def main():
    eng = ecgpu.Engine()
    rng = random.Random(7)
    for curve in ("k256", "p256"):
        c = pyref.CURVES[curve]
        n = 300
        ks = [rng.randrange(c.n) for _ in range(n)]; ks[0] = 0; ks[1] = c.n - 1
        pts = [pyref.mul(c, rng.randrange(1, c.n), pyref.G(c)) for _ in range(n)]; pts[2] = None
        xy, inf = pack_points(pts)
        oxy, oinf = eng.mul_batch(curve, pack_scalars(ks), xy, inf)
        got = unpack_points(oxy, oinf)
        for i in range(0, n, 37):
            assert got[i] == pyref.mul(c, ks[i], pts[i]), (curve, "mul", i)
        gxy, ginf = eng.mul_by_generator(curve, pack_scalars(ks))
        got = unpack_points(gxy, ginf)
        for i in range(0, n, 37):
            assert got[i] == pyref.mul(c, ks[i], pyref.G(c)), (curve, "gen", i)
        for m in (5, 8200):   # per-term path and bucket-method path (>= 2^13 terms)
            kk = [rng.randrange(c.n) for _ in range(m)]
            pp = [pts[i % n] for i in range(m)]
            pxy, pinf = pack_points(pp)
            lxy, linf = eng.lincomb(curve, pack_scalars(kk), pxy, pinf)
            rxy, rinf = ecref.lincomb(curve, pack_scalars(kk), pxy, pinf, nthreads=8)
            assert np.array_equal(np.asarray(lxy).reshape(-1), np.asarray(rxy).reshape(-1)) and int(linf) == int(rinf), (curve, "lincomb", m)
        a = [rng.randrange(c.n) for _ in range(n)]
        mxy, minf = eng.mul_by_generator_and_mul_add(curve, pack_scalars(a), pack_scalars(ks), xy, inf)
        got = unpack_points(mxy, minf)
        for i in range(0, n, 41):
            assert got[i] == pyref.add(c, pyref.mul(c, a[i], pyref.G(c)), pyref.mul(c, ks[i], pts[i])), (curve, "mga", i)
        fa = pack_scalars([rng.randrange(c.p) for _ in range(n)]); fb = pack_scalars([rng.randrange(c.p) for _ in range(n)])
        for op in range(6):
            eng.field_op(curve, op, fa, fb)
        sec1 = np.zeros((n, 33), np.uint8)
        for i, P in enumerate(pts):
            if P is not None:
                sec1[i, 0] = 2 + (P[1] & 1); sec1[i, 1:] = np.frombuffer(P[0].to_bytes(32, "big"), np.uint8)
        eng.decompress_batch(curve, sec1)
        # ECDSA
        z = np.frombuffer(os.urandom(32 * 64), np.uint8).reshape(64, 32).copy()
        sig = np.zeros((64, 64), np.uint8); q = np.zeros((64, 64), np.uint8)
        for i in range(64):
            d = rng.randrange(1, c.n)
            r, s = pyref.ecdsa_sign(c, d, int.from_bytes(z[i].tobytes(), "big"), rng.randrange(1, c.n))
            sig[i] = np.frombuffer(r.to_bytes(32, "big") + s.to_bytes(32, "big"), np.uint8)
            Q = pyref.mul(c, d, pyref.G(c)); q[i] = np.frombuffer(Q[0].to_bytes(32, "big") + Q[1].to_bytes(32, "big"), np.uint8)
        v = eng.ecdsa_verify_batch(curve, z, sig, q, low_s_only=False)
        assert v.all(), (curve, "ecdsa")
    # BIP340
    c = pyref.CURVES["k256"]
    pk = np.zeros((64, 32), np.uint8); msg = np.frombuffer(os.urandom(32 * 64), np.uint8).reshape(64, 32).copy(); sg = np.zeros((64, 64), np.uint8)
    for i in range(64):
        d = rng.randrange(1, c.n)
        px, s64 = pyref.bip340_sign(d, msg[i].tobytes(), os.urandom(32))
        pk[i] = np.frombuffer(px, np.uint8); sg[i] = np.frombuffer(s64, np.uint8)
        assert pyref.bip340_verify(px, msg[i].tobytes(), s64)
    assert eng.schnorr_verify_batch(pk, msg, sg).all()
    # SM2 public-key encryption: both entries, both layouts, both C1 forms, a refused record (empty message)
    c = pyref.CURVES["sm2"]
    d = rng.randrange(1, c.n); Pb = pyref.mul(c, d, pyref.G(c))
    pb = Pb[0].to_bytes(32, "big") + Pb[1].to_bytes(32, "big")
    msgs = [os.urandom(L) for L in (0, 1, 31, 32, 33, 56, 64, 65, 200, 1000)]
    kk = [rng.randrange(1, c.n) for _ in msgs]
    K = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in kk), np.uint8)
    for mode in (0, 1):
        for compressed in (True, False):
            cts, st = eng.sm2pke_encrypt_vartime(msgs, K, pb, mode, compressed)
            assert st.tolist() == [0] + [1] * 9, ("sm2pke", st)
            assert cts[3] == sm2pke_ref.sm2pke_encrypt(Pb, kk[3], msgs[3], mode, compressed)[1], ("sm2pke", "encrypt")
            assert eng.sm2pke_decrypt_vartime([x or b"" for x in cts], d.to_bytes(32, "big"), mode) == [None] + msgs[1:], ("sm2pke", "decrypt")
    eng.close()
    print("sanitize workload OK")

if __name__ == "__main__":
    main()
