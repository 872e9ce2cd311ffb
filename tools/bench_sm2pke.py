"""SM2 public-key encryption / decryption on one GPU (ecg_sm2pke_{encrypt,decrypt}_batch): prints one JSON line.

Shapes (each in both directions; one recipient key pair, as a server decrypting its queue holds one key):
  key_transport  2^18 records x 32-byte plaintexts
  hash_heavy     2^14 records x 4 KiB
  divergent      2^16 records, plaintext lengths uniform in 0-1024 (the empty ones are refused: status 0)
Per shape and direction:
  dev_ops_per_s      device-resident buffers (device-pointer mode), CUDA events around each call on the ctx's stream, a
                     256 MiB buffer written between timed calls (L2 flush; the working set then comes from HBM)
  e2e_ops_per_s      host (numpy) buffers in and out, host clock around the call (the call ends in a stream synchronise)
  scalar_mult_ms     per call, the scalar-multiplication kernels (ecg_timing_read: [d]C1, or [k]Pb and [k]G), and
  rest_ms            the rest of the device-resident call (front end, normalisation, KDF / C3 kernel, launches)
  bit_exact          every output byte (records, status / valid, pt_len) equal to the oracle pass
  cpu_baseline_s     duration of the oracle pass: scalar multiplications by the C restatement (oracle/ecref_prime.c) on all
                     host cores, then KDF / C3 / layout in Python (oracle/sm2pke_ref.py, hashlib's SM3 where present)
Usage: python tools/bench_sm2pke.py [--steps 5] [--warmup 2] [--scale 1] [--out FILE]   (--scale divides the record counts)
"""
import argparse
import hashlib
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "elliptic-curves_b200"), os.path.join(ROOT, "oracle")]
import ecgpu  # noqa: E402
import ecref  # noqa: E402
import pyref  # noqa: E402
import sm2pke_ref  # noqa: E402

C = pyref.CURVES["sm2"]
SM3 = (lambda b: hashlib.new("sm3", b).digest()) if "sm3" in hashlib.algorithms_available else sm2pke_ref.sm3
CORES = os.cpu_count() or 4


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return {"device": name, "power_limit_w": float(q[0]), "sm_max_mhz": float(q[1])}
    except Exception as e:  # noqa: BLE001
        return {"device": name, "power_limit_w": None, "error": str(e)[:100]}


def pack(recs):
    offs = np.zeros(len(recs) + 1, np.uint64)
    offs[1:] = np.cumsum([len(r) for r in recs], dtype=np.uint64)
    return np.frombuffer(b"".join(recs) + b"\0", np.uint8).copy(), offs


def oracle_encrypt(Pb, ks, msgs, mode, compressed):
    t0 = time.perf_counter()
    n = len(ks)
    K = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8).copy()
    PB = np.frombuffer((Pb[0].to_bytes(32, "big") + Pb[1].to_bytes(32, "big")) * n, np.uint8).copy()
    c1, _ = ecref.mul_gen_batch("sm2", K, nthreads=CORES)
    s, _ = ecref.mul_batch("sm2", K, PB, None, nthreads=CORES)
    c1, s = np.asarray(c1).reshape(n, 64), np.asarray(s).reshape(n, 64)
    ovh = 32 + (33 if compressed else 65)
    recs, status = [], np.zeros(n, np.uint8)
    for i, m in enumerate(msgs):
        if not m:
            recs.append(bytes(ovh))
            continue
        C1 = (int.from_bytes(c1[i, :32].tobytes(), "big"), int.from_bytes(c1[i, 32:].tobytes(), "big"))
        st, ct = sm2pke_ref.sm2pke_seal(C1, int.from_bytes(s[i, :32].tobytes(), "big"), int.from_bytes(s[i, 32:].tobytes(), "big"), m, mode,
                                   compressed, SM3)
        status[i] = st
        recs.append(ct if st == 1 else bytes(len(m) + ovh))
    return b"".join(recs), status, time.perf_counter() - t0


def oracle_decrypt(d, cts, mode):
    t0 = time.perf_counter()
    n = len(cts)
    parsed = [sm2pke_ref.sm2pke_parse(c, mode) for c in cts]
    D = np.frombuffer(d.to_bytes(32, "big") * n, np.uint8).copy()
    G = pyref.G(C)
    P = np.frombuffer(b"".join((p[0] if p else G)[0].to_bytes(32, "big") + (p[0] if p else G)[1].to_bytes(32, "big") for p in parsed), np.uint8).copy()
    s, _ = ecref.mul_batch("sm2", D, P, None, nthreads=CORES)
    s = np.asarray(s).reshape(n, 64)
    out, valid, pt_len = [], np.zeros(n, np.uint8), np.zeros(n, np.uint64)
    for i, (c, p) in enumerate(zip(cts, parsed)):
        m = None if p is None else sm2pke_ref.sm2pke_open(int.from_bytes(s[i, :32].tobytes(), "big"), int.from_bytes(s[i, 32:].tobytes(), "big"),
                                                     p[1], p[2], SM3)
        if m is not None:
            valid[i], pt_len[i] = 1, len(m)
        out.append((m or b"") + bytes(len(c) - len(m or b"")))
    return b"".join(out), valid, pt_len, time.perf_counter() - t0


def run_shape(name, n, lengths, args, info):
    import torch
    rng = random.Random(sum(name.encode()))
    msgs = [bytes(rng.getrandbits(8) for _ in range(L)) if L <= 64 else os.urandom(L) for L in lengths]
    d = rng.randrange(1, C.n)
    Pb = pyref.mul(C, d, pyref.G(C))
    ks = [rng.randrange(1, C.n) for _ in range(n)]
    K = np.frombuffer(b"".join(k.to_bytes(32, "big") for k in ks), np.uint8).copy()
    pb = np.frombuffer(Pb[0].to_bytes(32, "big") + Pb[1].to_bytes(32, "big"), np.uint8).copy()
    data, offs = pack(msgs)
    mode, compressed = 0, True
    res = {"n": n, "plaintext_bytes": int(offs[-1]), "mode": "c1c3c2", "c1": "compressed"}
    ref_ct, ref_st, t_enc = oracle_encrypt(Pb, ks, msgs, mode, compressed)
    host = ecgpu.Engine()
    dev = ecgpu.Engine(device_ptrs=True)
    stream = torch.cuda.current_stream()
    dev.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    g = torch.device("cuda:0")
    ovh = 32 + 33
    o_offs = (offs - offs[0]) + np.arange(n + 1, dtype=np.uint64) * np.uint64(ovh)
    t = {"data": torch.from_numpy(data).to(g), "offs": torch.from_numpy(offs.view(np.int64)).to(g), "k": torch.from_numpy(K).to(g),
         "pb": torch.from_numpy(np.tile(pb, n)).to(g), "ct": torch.zeros(int(o_offs[-1]) + 1, dtype=torch.uint8, device=g),
         "st": torch.zeros(n, dtype=torch.uint8, device=g), "ooffs": torch.from_numpy(o_offs.view(np.int64)).to(g),
         "d": torch.from_numpy(np.frombuffer(d.to_bytes(32, "big") * n, np.uint8).copy()).to(g),
         "pt": torch.zeros(int(o_offs[-1]) + 1, dtype=torch.uint8, device=g), "len": torch.zeros(n, dtype=torch.int64, device=g),
         "ok": torch.zeros(n, dtype=torch.uint8, device=g)}

    def enc_dev():
        dev.sm2pke_encrypt_ptr(n, t["data"].data_ptr(), t["offs"].data_ptr(), t["k"].data_ptr(), t["pb"].data_ptr(), mode, compressed,
                               t["ct"].data_ptr(), t["st"].data_ptr())

    def dec_dev():
        dev.sm2pke_decrypt_ptr(n, t["ct"].data_ptr(), t["ooffs"].data_ptr(), t["d"].data_ptr(), mode, t["pt"].data_ptr(), t["len"].data_ptr(),
                               t["ok"].data_ptr())

    def timed_dev(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        dev.timing_enable(True)
        ms = []
        for _ in range(args.steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        dom, calls = dev.timing_read()
        dev.timing_enable(False)
        med = float(np.median(ms))
        return {"dev_ms_median": med, "dev_ms_all": [round(x, 4) for x in ms], "dev_ops_per_s": n / (med / 1e3),
                "scalar_mult_ms": dom / max(calls, 1), "rest_ms": med - dom / max(calls, 1)}

    def timed_host(fn):
        for _ in range(args.warmup):
            fn()
        ws = []
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            ws.append(time.perf_counter() - t0)
        med = float(np.median(ws))
        return r, {"e2e_ms_median": med * 1e3, "e2e_ops_per_s": n / med}

    # encryption
    e = timed_dev(enc_dev)
    dev_ct = t["ct"].cpu().numpy()[:-1].tobytes()
    dev_st = t["st"].cpu().numpy()
    (h_ct, _, h_st), eh = timed_host(lambda: host.sm2pke_encrypt_packed_vartime(data, offs, K, pb, mode, compressed))
    e.update(eh)
    e["bit_exact"] = bool(dev_ct == ref_ct and h_ct.tobytes() == ref_ct and np.array_equal(dev_st, ref_st) and np.array_equal(h_st, ref_st))
    e["cpu_baseline_s"] = t_enc
    e["cpu_baseline_ops_per_s"] = n / t_enc
    e["refused"] = int((ref_st == 0).sum())
    res["encrypt"] = e
    # decryption of those ciphertexts
    cts = [ref_ct[int(o_offs[i]):int(o_offs[i + 1])] for i in range(n)]
    ref_pt, ref_ok, ref_len, t_dec = oracle_decrypt(d, cts, mode)
    dd = timed_dev(dec_dev)
    dev_pt = t["pt"].cpu().numpy()[:-1].tobytes()
    (h_pt, h_len, h_ok), dh = timed_host(lambda: host.sm2pke_decrypt_packed_vartime(np.frombuffer(ref_ct, np.uint8), o_offs, d.to_bytes(32, "big"), mode))
    dd.update(dh)
    dd["bit_exact"] = bool(dev_pt == ref_pt and h_pt.tobytes() == ref_pt and np.array_equal(t["ok"].cpu().numpy(), ref_ok) and
                           np.array_equal(h_ok, ref_ok) and np.array_equal(t["len"].cpu().numpy().astype(np.uint64), ref_len) and
                           np.array_equal(h_len, ref_len))
    dd["cpu_baseline_s"] = t_dec
    dd["cpu_baseline_ops_per_s"] = n / t_dec
    dd["valid"] = int(ref_ok.sum())
    res["decrypt"] = dd
    host.close()
    dev.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=int, default=1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_sm2pke: no CUDA device (this benchmark measures the GPU; there is no CPU fallback)")
    info = gpu_info()
    rng = random.Random(3)
    shapes = {"key_transport": ((1 << 18) // args.scale, lambda n: [32] * n),
              "hash_heavy": ((1 << 14) // args.scale, lambda n: [4096] * n),
              "divergent": ((1 << 16) // args.scale, lambda n: [rng.randrange(0, 1025) for _ in range(n)])}
    out = {"bench": "sm2pke", **info, "host_cores": CORES, "steps": args.steps, "warmup": args.warmup, "shapes": {}}
    for name, (n, lens) in shapes.items():
        out["shapes"][name] = run_shape(name, n, lens(n), args, info)
    out["bit_exact"] = all(s[d]["bit_exact"] for s in out["shapes"].values() for d in ("encrypt", "decrypt"))
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
