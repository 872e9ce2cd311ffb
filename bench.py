#!/usr/bin/env python3
"""bench.py — the measurement contract for the batched scalar-multiplication hot path.

    python bench.py --gpus N --steps K --warmup W            # our arm  (libecgpu.so, sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the CPU restatement of the
                                                             # reference's own algorithm on the host cores
  N > 1 is launched by `python -m torch.distributed.run --nproc-per-node N ...` (one rank per GPU).
  --dump-outputs DIR writes what the headline's last timed step computed (see dump_outputs); the inputs are seeded, so two
  builds run with the same arguments can be compared output for output.

A "step" = one pass of the hot path over one batch: BASELINE.json configs[1], secp256k1 variable-base
scalar multiplication of 2^20 (scalar, point) pairs per GPU (weak scaling: each rank owns its own 2^20 pairs,
no data-path collective).  Other workloads (--workload) are the remaining BASELINE configs; they print the
same JSON line but are not the headline.

Timed regions
  value : inputs/outputs resident in HBM (ECG_FLAG_DEVICE_PTRS), CUDA events on the launching stream,
          K steps between barrier+synchronize, max over ranks.
  e2e   : same metric through the host-buffer C ABI call: pinned host inputs -> H2D -> kernels -> D2H of the
          affine results inside the timed region.
  roofline / cpu_baseline : see DESIGN.md section "Measurement".
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "elliptic-curves_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np

WORKLOADS = {
    # name: (curve, op, log2 batch per GPU, BASELINE.json config index, unit noun)
    "k256_varbase": ("k256", "mul", 20, 1, "scalar-mults/s"),
    "p256_varbase": ("p256", "mul", 20, 2, "scalar-mults/s"),
    "k256_fixedbase": ("k256", "mulgen", 22, 3, "scalar-mults/s"),
    "k256_lincomb": ("k256", "lincomb", 21, 4, "terms/s"),
    # first widening step (SURVEY 8(f) rank 1), not a BASELINE.json config: BIP340 verification
    "k256_schnorr_verify": ("k256", "schnorr", 20, None, "verifications/s"),
}
SEEDS = {"k256_varbase": 0xB2000001, "p256_varbase": 0xB2000002, "k256_fixedbase": 0xB2000003, "k256_lincomb": 0xB2000004,
         "k256_schnorr_verify": 0xB2000005}
ALGO_BYTES = {"mul": 160, "mulgen": 96, "lincomb": 96, "schnorr": 129}  # SURVEY.md section 8(d): algorithmic bytes per unit
# IMAD.WIDE (32x32->64 multiply-accumulate) instructions per unit of work in the dominant kernel, counted from
# the kernels' operation schedule (derivation: DESIGN.md "Integer roofline"):
#   k256: M = 64 + 8 (product + reduction), S = 36 + 8;  var-base = 1046 M + 748 S + 129 mul_small*8 + GLV ~200
#   p256: M = 64, S = 36 (Solinas reduction uses no multiplier); var-base = 1885 M + 1316 S + 258*8
#   k256 fixed-base: 17 mixed additions = 136 M + 51 S
#   k256 lincomb (bucket kernel, c = 16): 2 halves x 8 windows mixed additions = 128 M + 48 S per term
#   k256 schnorr verify (mul_gen_add kernel): var-base + fixed-base accumulation
# SURVEY.md section 8(d): the graded roofline of this path is the integer multiply-add issue rate; its canonical
# ALGORITHMIC work per unit (one "IMAD" = one 32x32->64 multiply-accumulate = one IMAD.WIDE on sm_100a):
SURVEY_IMAD_PER_UNIT = {("k256", "mul"): 1.47e5, ("p256", "mul"): 2.30e5, ("k256", "mulgen"): 2.9e4, ("k256", "lincomb"): 1.5e4,
                        ("k256", "schnorr"): 1.47e5 + 2.9e4}
# what the kernels actually execute (fewer products than the canonical model: dedicated squaring, 16-bit fixed-base
# windows, bucket method):
IMADW_PER_UNIT = {("k256", "schnorr"): 121_500, ("k256", "mul"): 109_500, ("p256", "mul"): 170_100, ("k256", "mulgen"): 12_000, ("k256", "lincomb"): 11_300}


def synth_scalars(curve, seed, start, count):
    """k_i = SHA-256(seed || "k" || LE64(i)) mod n   (SURVEY.md section 8(d))"""
    import pyref

    n = pyref.CURVES[curve].n
    out = bytearray(32 * count)
    pre = seed.to_bytes(8, "little")
    for j in range(count):
        i = start + j
        h = hashlib.sha256(pre + b"k" + i.to_bytes(8, "little")).digest()
        v = int.from_bytes(h, "big")
        if v >= n:
            v -= n
        out[32 * j:32 * j + 32] = v.to_bytes(32, "big")
    return np.frombuffer(bytes(out), dtype=np.uint8).copy()


def synth_point_scalars(curve, seed, start, count):
    """t_i = SHA-256(seed || "p" || LE64(i)) mod n, t_i != 0 ; P_i = t_i * G"""
    import pyref

    n = pyref.CURVES[curve].n
    out = bytearray(32 * count)
    pre = seed.to_bytes(8, "little")
    for j in range(count):
        i = start + j
        h = hashlib.sha256(pre + b"p" + i.to_bytes(8, "little")).digest()
        v = int.from_bytes(h, "big") % n
        if v == 0:
            v = 1
        out[32 * j:32 * j + 32] = v.to_bytes(32, "big")
    return np.frombuffer(bytes(out), dtype=np.uint8).copy()


def synth_schnorr(eng, seed, start, count):
    """count valid BIP340 (pk, msg, sig) triples: keys and nonces from the seeded hash, k*G / d*G on the GPU's
    fixed-base path, challenges with hashlib, s = k + e*d on the host."""
    import pyref

    c = pyref.K256
    n, p = c.n, c.p
    d = synth_point_scalars("k256", seed, start, count)
    k = synth_scalars("k256", seed ^ 0x5A5A, start, count)
    Pxy, _ = eng.mul_by_generator("k256", d)
    Rxy, Rinf = eng.mul_by_generator("k256", k)
    Pxy, Rxy = np.asarray(Pxy).reshape(count, 64), np.asarray(Rxy).reshape(count, 64)
    pk = np.ascontiguousarray(Pxy[:, :32]).reshape(-1)
    msg = synth_scalars("k256", seed ^ 0xA5A5, start, count)  # any 32 bytes
    sig = np.empty((count, 64), np.uint8)
    th = hashlib.sha256(b"BIP0340/challenge").digest()
    pre = hashlib.sha256(th + th)
    dv, kv, mv = d.reshape(count, 32), k.reshape(count, 32), msg.reshape(count, 32)
    for i in range(count):
        di = int.from_bytes(dv[i].tobytes(), "big")
        ki = int.from_bytes(kv[i].tobytes(), "big")
        if ki == 0 or Rinf[i]:
            ki = 1
        if Pxy[i, 63] & 1:
            di = n - di
        if Rxy[i, 63] & 1:
            ki = n - ki
        h = pre.copy()
        h.update(Rxy[i, :32].tobytes() + Pxy[i, :32].tobytes() + mv[i].tobytes())
        e = int.from_bytes(h.digest(), "big") % n
        sig[i, :32] = Rxy[i, :32]
        sig[i, 32:] = np.frombuffer(((ki + e * di) % n).to_bytes(32, "big"), np.uint8)
    return pk, msg, sig.reshape(-1)


def host_cores():
    """(usable cores, how we know): the affinity mask capped by the cgroup CPU quota (the GPU boxes expose 128
    logical CPUs but give the container 16 cores' worth of time; oversubscribing them only adds throttling)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    why = "sched_getaffinity"
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            c = max(1, int(float(q) / float(per) + 0.5))
            if c < n:
                n, why = c, f"cgroup cpu.max {q}/{per}"
    except (OSError, ValueError):
        pass
    return n, why


def best_thread_count(fn, cores):
    """Give the CPU arm its best shot: time a small sample at 1x and 2x the usable cores, keep the faster."""
    best, best_t = cores, None
    for nt in (cores, 2 * cores):
        t0 = time.perf_counter()
        fn(nt)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    return best


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def mark(self):
        """index of the next sample (call at the start / end of the timed region)"""
        return len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self, lo=0, hi=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        rows = self.rows[lo:hi] if (hi is not None and hi - lo >= 3) else self.rows
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": max(mx), "power_w_max": max(power), "samples": len(sm), "reasons": sorted(reasons)}


DUMP_ROWS = 1 << 17   # per-element outputs larger than this are dumped as a fixed sample of rows (<= 34 MB in all)
DUMP_SEED = 0xB2000D00


def dump_outputs(out_dir, op, n, out_xy, out_inf):
    """Write what one step of the timed path returned to its caller as float32 .npy files (byte values 0..255, exact):
    mul / mulgen -> xy [rows, 64] (big-endian x || y) + inf [rows]; lincomb -> the one sum point; schnorr -> valid [rows].
    Batches above DUMP_ROWS are sampled at fixed, seeded row indices (index.npy), so two builds can be compared row for row."""
    os.makedirs(out_dir, exist_ok=True)
    if op == "lincomb":
        arrays = {"xy": out_xy.reshape(1, 64), "inf": out_inf[:1]}
    else:
        idx = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))
        arrays = {"index": idx}
        if op == "schnorr":
            arrays["valid"] = out_xy[idx]
        else:
            arrays["xy"] = out_xy.reshape(n, 64)[idx]
            arrays["inf"] = out_inf[idx]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))
    return sorted(arrays)


def dist_setup(n_gpus):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(local)
    return world, rank, local


def barrier_sync(world):
    import torch

    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch

    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


class Bench:
    """What every measured config shares on this rank: engines, L2-flush buffer, integer peak, host core budget."""

    def __init__(self, args):
        import torch

        import ecgpu

        self.args = args
        self.world, self.rank, self.local = dist_setup(args.gpus)
        self.dev = torch.device("cuda", self.local)
        self.host_eng = ecgpu.Engine([self.local])                       # host-buffer ABI (e2e)
        self.eng = ecgpu.Engine([self.local], device_ptrs=True)          # device-resident ABI (value)
        self.eng.set_stream(torch.cuda.current_stream().cuda_stream)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
        self.imadw_peak, _ = self.eng.microbench(0, 4000)                # IMAD.WIDE issue rate, this GPU, this run
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            self.hbm_peak, self.hbm_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
        else:
            self.hbm_peak, self.hbm_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
        self.traffic = {}
        for name in ("r02_traffic.json", "r01_traffic.json"):
            prof = os.path.join(ROOT, "profiles", name)
            if os.path.exists(prof):
                for k, v in json.load(open(prof)).items():
                    self.traffic.setdefault(k, v)
        # host cores: the cgroup quota is shared by all ranks of the job; every rank checks its own outputs with its share
        import ecref

        self.cores, self.cores_why = host_cores()
        k_probe = synth_scalars("k256", 1, 0, 4096)
        self.threads_total = best_thread_count(lambda nt: ecref.mul_gen_batch("k256", k_probe, nthreads=max(1, nt // self.world)), self.cores)
        self.threads = max(1, self.threads_total // self.world)

    def all_true(self, flag):
        """logical AND of a per-rank boolean"""
        import torch

        if self.world == 1:
            return bool(flag)
        import torch.distributed as dist

        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def sum_over_ranks(self, x):
        import torch

        if self.world == 1:
            return x
        import torch.distributed as dist

        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())


def measure(B, workload, steps, warmup, sample_clocks, dump_dir=None):
    """One BASELINE config on this job's ranks: device-resident rate (`value`), end-to-end rate through the host-buffer ABI,
    bit-exact comparison of EVERY output with the CPU restatement, roofline.  Returns the record on rank 0, None elsewhere.
    dump_dir: rank 0 writes the device path's outputs of the last timed step there (dump_outputs)."""
    import torch

    import ecref
    import pyref

    args, world, rank, dev, eng, host_eng = B.args, B.world, B.rank, B.dev, B.eng, B.host_eng
    curve, op, logn, cfg_idx, unit = WORKLOADS[workload]
    if args.log2_batch:
        logn = args.log2_batch
    n = 1 << logn
    seed = SEEDS[workload]
    start = rank * n

    # ---- synthetic inputs: scalars hashed on the host, points P_i = t_i*G made with the fixed-base kernel
    a_host = None
    if op == "schnorr":
        pk_np, msg_np, sig_np = synth_schnorr(host_eng, seed, start, n)
        k_host = torch.from_numpy(pk_np).pin_memory()      # pk  (32 B)
        a_host = torch.from_numpy(msg_np).pin_memory()     # msg (32 B)
        p_host = torch.from_numpy(sig_np).pin_memory()     # sig (64 B)
    else:
        k_host = torch.from_numpy(synth_scalars(curve, seed, start, n)).pin_memory()
        if op != "mulgen":
            t_host = synth_point_scalars(curve, seed, start, n)
            pxy, pinf = host_eng.mul_by_generator(curve, t_host)
            assert not pinf.any()
            p_host = torch.from_numpy(np.ascontiguousarray(pxy).reshape(-1)).pin_memory()
        else:
            p_host = None
    out_bytes = {"lincomb": 64, "schnorr": n}.get(op, 64 * n)
    n_inf = n if op != "lincomb" else 1
    out_host = torch.empty(out_bytes, dtype=torch.uint8).pin_memory()
    oinf_host = torch.empty(n_inf, dtype=torch.uint8).pin_memory()
    kd = k_host.to(dev)
    pd = p_host.to(dev) if p_host is not None else None
    ad = a_host.to(dev) if a_host is not None else None
    oxy = torch.zeros(out_bytes, dtype=torch.uint8, device=dev)
    oinf = torch.zeros(n_inf, dtype=torch.uint8, device=dev)
    part_d = torch.empty(96, dtype=torch.uint8, device=dev)
    parts_d = torch.empty(96 * world, dtype=torch.uint8, device=dev)
    exchange = op == "lincomb" and world > 1
    if exchange:
        import torch.distributed as dist

    def step_dev(with_exchange=True):
        B.flush.zero_()  # L2 flush between timed iterations
        if op == "mul":
            eng.mul_batch_ptr(curve, n, kd.data_ptr(), pd.data_ptr(), 0, oxy.data_ptr(), oinf.data_ptr())
        elif op == "mulgen":
            eng.mul_gen_batch_ptr(curve, n, kd.data_ptr(), oxy.data_ptr(), oinf.data_ptr())
        elif op == "schnorr":
            eng.schnorr_verify_ptr(n, kd.data_ptr(), ad.data_ptr(), pd.data_ptr(), oxy.data_ptr())
        elif not (exchange and with_exchange):
            eng.lincomb_ptr(curve, n, kd.data_ptr(), pd.data_ptr(), 0, oxy.data_ptr(), oinf.data_ptr())
        else:
            # config 5: every rank reduces its 2^21 terms to one Jacobian point; ONE exchange step (all_gather of 96 bytes
            # per rank over NCCL/NVLink); rank 0 adds the `world` partial points where the all_gather left them and
            # normalises — nothing of the exchange touches the host
            eng.lincomb_partial_ptr(curve, n, kd.data_ptr(), pd.data_ptr(), 0, part_d.data_ptr())
            dist.all_gather_into_tensor(parts_d, part_d)
            if rank == 0:
                eng.point_sum_ptr(curve, world, parts_d.data_ptr(), oxy.data_ptr(), oinf.data_ptr())

    def step_host():
        k_np, o_np, oi_np = k_host.numpy(), out_host.numpy(), oinf_host.numpy()
        if op == "mul":
            host_eng.mul_batch(curve, k_np, p_host.numpy(), None, o_np, oi_np)
        elif op == "mulgen":
            host_eng.mul_by_generator(curve, k_np, o_np, oi_np)
        elif op == "schnorr":
            o_np[:] = host_eng.schnorr_verify_batch(k_np, a_host.numpy(), p_host.numpy())
        elif not exchange:
            xy, inf = host_eng.lincomb(curve, k_np, p_host.numpy(), None)
            o_np[:] = xy
            oi_np[0] = inf
        else:
            part = host_eng.lincomb_partial(curve, k_np, p_host.numpy(), None)   # H2D of this rank's terms inside
            part_d.copy_(torch.from_numpy(part), non_blocking=False)
            dist.all_gather_into_tensor(parts_d, part_d)
            if rank == 0:
                eng.point_sum_ptr(curve, world, parts_d.data_ptr(), oxy.data_ptr(), oinf.data_ptr())
                o_np[:] = oxy.cpu().numpy()                                   # D2H of the result
                oi_np[0] = int(oinf.cpu()[0])

    def timed(fn, k):
        barrier_sync(world)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(k):
            fn()
        ev1.record()
        barrier_sync(world)
        return max_over_ranks(ev0.elapsed_time(ev1), world)

    # ---- device-resident timing (the `value`)
    sampler = ClockSampler(B.local) if (rank == 0 and sample_clocks) else None
    if sampler:
        sampler.start()
    for _ in range(max(warmup, 3)):
        step_dev()
    eng.timing_enable(True)
    launches0 = eng.kernel_launches
    m0 = sampler.mark() if sampler else 0
    ms_total = timed(step_dev, steps)
    clocks = sampler.stop(m0, sampler.mark()) if sampler else None
    launches = eng.kernel_launches - launches0
    dom_ms, dom_calls = eng.timing_read()
    eng.timing_enable(False)
    ms_per_step = ms_total / steps
    value = world * n * steps / (ms_total * 1e-3)
    dev_xy, dev_inf = oxy.cpu().numpy().copy(), oinf.cpu().numpy().copy()
    dumped = dump_outputs(dump_dir, op, n, dev_xy, dev_inf) if (dump_dir and rank == 0) else None
    exch = None
    if exchange:
        # the same call without the exchange step (every rank reduces and normalises its own terms): what the NCCL
        # exchange + the device-side point sum add to a step, measured in the same run
        for _ in range(2):
            step_dev(False)
        ms_local = timed(lambda: step_dev(False), steps) / steps
        exch = {"ms_per_step_with_exchange": ms_per_step, "ms_per_step_local_only": ms_local,
                "exchange_efficiency": ms_local / ms_per_step,
                "what": "all_gather_into_tensor of 96 B per rank (NCCL) + ecg_point_sum on rank 0 straight from the receive buffer"}

    # ---- end-to-end through the host-buffer ABI (pinned host memory, H2D + D2H inside the timed region)
    for _ in range(2):
        step_host()
    barrier_sync(world)
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host()
    barrier_sync(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    e2e_value = world * n * steps / e2e_s
    h2d = 32 * n + (64 * n if op != "mulgen" else 0) + (32 * n if op == "schnorr" else 0)
    d2h = {"lincomb": 65, "schnorr": n}.get(op, 65 * n)
    if exchange:
        same = True if rank != 0 else bool(np.array_equal(dev_xy, out_host.numpy()) and dev_inf[0] == oinf_host.numpy()[0])
    elif op == "schnorr":
        same = bool(np.array_equal(dev_xy, out_host.numpy())) and bool(out_host.numpy().all())
    else:
        same = bool(np.array_equal(dev_xy, out_host.numpy())) and bool(np.array_equal(dev_inf, oinf_host.numpy()))
    same = B.all_true(same)

    # ---- parity: EVERY output of this rank against the CPU restatement (oracle/ecref.c, constant-time `*` path), on this
    #      rank's share of the host cores, outside the timed regions.  Its duration is the CPU baseline of this config.
    nt = B.threads
    barrier_sync(world)
    t0 = time.perf_counter()
    if op == "schnorr":
        # the reference's verify_raw = tagged hash + mul_by_generator_and_mul_add_vartime(s, -e, P) + checks; the CPU leg
        # times the group-operation part on a sample; validity itself is known by construction (every signature is valid)
        ns = min(n, 1 << 16)
        s_s = np.ascontiguousarray(p_host.numpy().reshape(n, 64)[:ns, 32:]).reshape(-1)
        pxy_s, _ = host_eng.mul_by_generator(curve, synth_point_scalars(curve, seed, start, ns))
        t0 = time.perf_counter()
        ecref.mul_gen_add_batch(curve, s_s, k_host.numpy()[:32 * ns], np.asarray(pxy_s).reshape(-1), None, nthreads=nt)
        cpu_units, bit_exact = ns, bool(out_host.numpy().all())
    elif op == "mul":
        r_xy, r_inf = ecref.mul_batch(curve, k_host.numpy(), p_host.numpy(), None, nthreads=nt, variant=0)
        cpu_units, bit_exact = n, bool(np.array_equal(out_host.numpy(), r_xy.reshape(-1)) and np.array_equal(oinf_host.numpy(), r_inf))
    elif op == "mulgen":
        r_xy, r_inf = ecref.mul_gen_batch(curve, k_host.numpy(), nthreads=nt)
        cpu_units, bit_exact = n, bool(np.array_equal(out_host.numpy(), r_xy.reshape(-1)) and np.array_equal(oinf_host.numpy(), r_inf))
    else:
        r_xy, r_inf = ecref.lincomb(curve, k_host.numpy(), p_host.numpy(), None, nthreads=nt)   # this rank's terms
        cpu_units = n
        if not exchange:
            bit_exact = bool(np.array_equal(out_host.numpy(), r_xy) and int(oinf_host.numpy()[0]) == r_inf)
    cpu_s = time.perf_counter() - t0
    if exchange:
        # the oracle's per-rank sums travel to rank 0 (65 bytes each), which adds them with the big-integer model and
        # compares with the GPU job's global result: 100 % of the 2^21 * world terms are covered
        mine = torch.from_numpy(np.concatenate([r_xy.reshape(-1), np.array([r_inf], np.uint8)])).to(dev)
        allp = torch.empty(65 * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allp, mine)
        bit_exact = True
        if rank == 0:
            c = pyref.CURVES[curve]
            acc = None
            for r in range(world):
                rec = allp[65 * r:65 * r + 65].cpu().numpy()
                acc = pyref.add(c, acc, pyref.dec_point(rec[:64].tobytes(), int(rec[64])))
            exp_xy, exp_inf = pyref.enc_point(acc)
            bit_exact = bool(out_host.numpy().tobytes() == exp_xy and int(oinf_host.numpy()[0]) == exp_inf
                             and dev_xy.tobytes() == exp_xy and int(dev_inf[0]) == exp_inf)
    bit_exact = B.all_true(bit_exact)
    cpu_rate = B.sum_over_ranks(cpu_units / cpu_s)

    if rank != 0:
        return None
    dom_avg_ms = dom_ms / max(dom_calls, 1)
    achieved_gbs = ALGO_BYTES[op] * n / (dom_avg_ms * 1e-3) / 1e9
    imadw_unit = IMADW_PER_UNIT.get((curve, op))
    roofline_int = None
    if imadw_unit:
        ach = imadw_unit * n / (dom_avg_ms * 1e-3)
        roofline_int = {"bound": "int32 multiply issue (IMAD.WIDE.U32 on the fmaheavy pipe, 4 cycles per warp instruction)", "achieved": ach,
                        "peak": B.imadw_peak, "unit": "IMAD.WIDE/s (executed)", "frac": ach / B.imadw_peak, "imad_wide_per_unit": imadw_unit,
                        "peak_source": "ecg_microbench(0) in this run; independent record: profiles/r02_ncu_mb_imad_wide.json (fmaheavy 95.3 % busy)"}
    survey_unit = SURVEY_IMAD_PER_UNIT.get((curve, op))
    ach_alg = survey_unit * n / (dom_avg_ms * 1e-3)
    covered = "every output" if op != "schnorr" else "every verdict (all signatures valid by construction)"
    rec = {
        "metric": "scalar-mults/sec (var-base, batch) at 1/2/4/8 B200 vs reference Rust CPU" if op == "mul" and curve == "k256" else f"{unit} ({workload})",
        "value": value, "unit": unit, "n_gpus": world, "steps": steps, "warmup": max(warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": (f"BASELINE.json configs[{cfg_idx}]: " if cfg_idx is not None else "widening step (not a BASELINE config): ")
                               + f"{workload}, batch 2^{logn} per GPU", "curve": curve,
                   "batch_per_gpu": n, "inputs": "k_i, t_i = SHA-256(seed||tag||LE64(i)) mod n; P_i = t_i*G (SURVEY 8(d))",
                   "l2": "256 MiB buffer written between timed iterations (L2 flush); working set > L2",
                   "parallelism": (f"terms sharded over {world} rank(s); one exchange step: all_gather of 96 B per rank over NCCL, "
                                   "device-side sum of the partial points on rank 0" if exchange else
                                   f"batch sharded over {world} rank(s), no data-path collective")},
        "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "note": "host-buffer C ABI call, pinned host memory, copies inside the timed region", "matches_device_path": same},
        "gpu_launches": launches,
        "bit_exact": bit_exact,
        "bit_exact_coverage": f"{covered} of every rank vs the CPU restatement (oracle/ecref.c), {world * cpu_units} units",
        # SURVEY.md section 8(d): "neither HBM nor tensor cores - the INT32 multiply-add issue rate"; achieved =
        # algorithmic IMADs per unit (SURVEY's canonical model) x units / dominant-kernel time; peak = IMAD.WIDE
        # issue rate measured live by ecg_microbench(0) (MEASURED_PEAKS.json has no integer peak)
        "roofline": {"bound": "int32-imad", "achieved": ach_alg, "peak": B.imadw_peak, "unit": "IMAD/s", "frac": ach_alg / B.imadw_peak,
                     "traffic": B.traffic.get(workload), "kernel_ms": dom_avg_ms, "imad_per_unit": survey_unit,
                     "model": "SURVEY.md 8(d) canonical algorithmic count; peak = measured IMAD.WIDE.U32 issue rate (this run)",
                     "note": ("SURVEY's canonical model counts more multiply-adds per unit than this kernel executes "
                              f"({survey_unit:.3g} vs {imadw_unit or 0:.3g}); frac is therefore an algorithmic-throughput ratio and can "
                              "approach or exceed 1. roofline_int is the fraction of the multiplier's issue rate actually used.")},
        "roofline_int": roofline_int,
        "roofline_hbm": {"bound": "hbm", "achieved": achieved_gbs, "peak": B.hbm_peak, "unit": "GB/s", "frac": achieved_gbs / B.hbm_peak,
                         "peak_source": B.hbm_src, "algorithmic_bytes_per_unit": ALGO_BYTES[op],
                         "note": "reported because north_star asks for it; this path is not HBM bound"},
        "cpu_baseline": {"value": cpu_rate, "unit": unit, "cores": B.cores, "threads": B.threads * world, "cores_source": B.cores_why, "kind": "port",
                         "sample": (f"the whole workload ({world * cpu_units} units), constant-time `*` path (oracle/ecref.c), "
                                    f"{B.threads} thread(s) per rank x {world} rank(s) on {B.cores} usable cores; the same pass is the parity check"),
                         "bit_exact_vs_gpu": bit_exact},
    }
    if clocks is not None:
        rec["clocks"] = clocks
    if dumped is not None:
        rec["dumped_outputs"] = {"dir": os.path.abspath(dump_dir), "arrays": dumped, "rank": 0}
    if exch is not None:
        rec["exchange"] = exch
    return rec


def config1_plumbing(B):
    """BASELINE.json configs[0] / BASELINE.md section 3 row 1: single-thread latencies of the reference's benchmarked
    operations (k256/benches/point.rs:62-104) on the CPU restatement, and the restatement's results on the reference's
    own vectors.  No GPU in this record."""
    import ecref
    import pyref
    from helpers import golden

    out = {"workload": "BASELINE.json configs[0]: k256 ProjectivePoint::mul, scalar x G on CPU (plumbing)", "kind": "port", "threads": 1}
    for curve in ("k256", "p256"):
        c = pyref.CURVES[curve]
        g = golden(curve)
        ks = np.frombuffer(b"".join(bytes.fromhex(v["k"]) for v in g["group"]["mul"]), np.uint8)
        want = b"".join(bytes.fromhex(v["x"]) + bytes.fromhex(v["y"]) for v in g["group"]["mul"])
        Gxy, _ = pyref.enc_point(pyref.G(c))
        m = ks.size // 32
        Pg = np.frombuffer(Gxy * m, np.uint8)
        ok = ecref.mul_gen_batch(curve, ks, nthreads=1)[0].tobytes() == want
        ok = ok and ecref.mul_batch(curve, ks, Pg, None, nthreads=1, variant=0)[0].tobytes() == want
        ok = ok and ecref.mul_batch(curve, ks, Pg, None, nthreads=1, variant=1)[0].tobytes() == want
        # the bench scalars of k256/benches/point.rs:18-40 (and the P-256 twins), repeated: single-thread rate -> latency
        bs = [bytes.fromhex(v["k"]) for v in g["bench"]["scalars"]]
        reps = 1500
        kk = np.frombuffer(b"".join(bs[i % len(bs)] for i in range(reps)), np.uint8)
        PP = np.frombuffer(Gxy * reps, np.uint8)
        lat = {}
        for name, fn in (("mul (constant-time `*`)", lambda: ecref.mul_batch(curve, kk, PP, None, nthreads=1, variant=0)),
                         ("mul_vartime", lambda: ecref.mul_batch(curve, kk, PP, None, nthreads=1, variant=1)),
                         ("mul_by_generator", lambda: ecref.mul_gen_batch(curve, kk, nthreads=1)),
                         ("lincomb (2 terms)", lambda: [ecref.lincomb(curve, kk[:64], PP[:128], None, nthreads=1) for _ in range(300)])):
            fn()
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            lat[name] = {"us_per_op": dt / (300 if name.startswith("lincomb") else reps) * 1e6}
        out[curve] = {"golden_mul_vectors": m, "golden_ok": bool(ok), "single_thread_latency": lat}
    return out


def strong_scaling(B):
    """One host-resident batch of 2^LOG pairs held by rank 0, split over the job's GPUs two ways:
       (a) NCCL: rank 0 uploads everything over ITS PCIe link, scatter / gather over NVLink (ecgpu.dist),
       (b) one multi-device ecg_ctx in rank 0's process: every GPU pulls its slice over its own PCIe link.
    Both are timed end to end (host buffers in, host buffers out); the results must be identical."""
    import torch
    import torch.distributed as dist

    import ecgpu
    import ecref
    from ecgpu import dist as ecdist

    world, rank = B.world, B.rank
    logn = B.args.strong_log2
    n = 1 << logn
    rec = None
    k = pxy = None
    if rank == 0:
        rng = np.random.default_rng(0xB2000006)
        k = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        k[:, 0] &= 0x7F   # < 2^255 < n
        t = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        t[:, 0] &= 0x7F
        t[:, 31] |= 1     # non-zero
        pxy, pinf = B.host_eng.mul_by_generator("k256", t.reshape(-1))
        k = torch.from_numpy(k.reshape(-1)).pin_memory().numpy()
        pxy = torch.from_numpy(np.ascontiguousarray(pxy).reshape(-1)).pin_memory().numpy()
    reps = 3
    times_a = []
    out_a = None
    a_xy = torch.empty(64 * n, dtype=torch.uint8).pin_memory().numpy() if rank == 0 else None
    a_inf = torch.empty(n, dtype=torch.uint8).pin_memory().numpy() if rank == 0 else None
    for it in range(reps + 1):
        barrier_sync(world)
        t0 = time.perf_counter()
        out_a = ecdist.mul_batch_distributed(B.eng, "k256", n, k, pxy, src=0, out_xy=a_xy, out_inf=a_inf)
        barrier_sync(world)
        if it:
            times_a.append(time.perf_counter() - t0)
    times_b = []
    out_b = None
    if rank == 0:
        md = ecgpu.Engine(list(range(world)))
        oxy = torch.empty(64 * n, dtype=torch.uint8).pin_memory().numpy()
        oinf = torch.empty(n, dtype=torch.uint8).pin_memory().numpy()
        for it in range(reps + 1):
            t0 = time.perf_counter()
            md.mul_batch("k256", k, pxy, None, oxy, oinf)
            if it:
                times_b.append(time.perf_counter() - t0)
        out_b = (oxy, oinf)
        md.close()
    barrier_sync(world)
    if rank == 0:
        same = bool(np.array_equal(out_a[0], out_b[0]) and np.array_equal(out_a[1], out_b[1]))
        ns = min(n, 1 << 17)
        r_xy, r_inf = ecref.mul_batch("k256", np.concatenate([k[:32 * ns], k[-32 * ns:]]), np.concatenate([pxy[:64 * ns], pxy[-64 * ns:]]), None,
                                      nthreads=B.threads_total, variant=0)
        got = np.concatenate([out_b[0][:64 * ns], out_b[0][-64 * ns:]])
        ok = bool(np.array_equal(got, r_xy.reshape(-1)))
        ta, tb = min(times_a), min(times_b)
        rec = {"workload": f"k256 var-base, ONE batch of 2^{logn} pairs in rank 0's pinned host memory, {world} GPUs (strong scaling)",
               "nccl_scatter_gather": {"mults_per_s": n / ta, "ms": ta * 1e3,
                                       "path": "rank 0 H2D (one PCIe link) -> dist.scatter over NVLink -> kernels -> dist.gather -> rank 0 D2H"},
               "multi_device_ctx": {"mults_per_s": n / tb, "ms": tb * 1e3,
                                    "path": "one ecg_ctx over all GPUs in rank 0's process: every GPU copies its own slice over its own PCIe link"},
               "bytes_over_rank0_pcie": {"nccl": 161 * n, "multi_device_ctx": 161 * n // world},
               "limiter": "rank 0's PCIe link for the NCCL variant (all 161 B/pair cross it); per-GPU PCIe + the host memory system for the multi-device ctx",
               "results_identical": same, "bit_exact_sample": ok,
               "bit_exact_coverage": f"first and last 2^{ns.bit_length() - 1} pairs vs oracle/ecref.c; (a) == (b) on all 2^{logn} outputs"}
    return rec


def multi_device_parity(B):
    """tests/test_gpu_parity.py::test_multi_device_ctx_shards_the_batch needs >= 2 GPUs, which the 1-GPU test box does not
    have: the same check runs here whenever the bench is launched on several GPUs (rank 0, every visible device)."""
    import ecgpu
    import ecref

    n = 5003
    k = synth_scalars("k256", 0xB2000007, 0, n)
    t = synth_point_scalars("k256", 0xB2000007, 0, n)
    pxy, _ = B.host_eng.mul_by_generator("k256", t)
    pxy = np.ascontiguousarray(pxy).reshape(-1)
    md = ecgpu.Engine(list(range(B.world)))
    res = {}
    for curve in ("k256",):
        oxy, oinf = md.mul_batch(curve, k, pxy)
        r_xy, r_inf = ecref.mul_batch(curve, k, pxy, None, nthreads=B.threads_total, variant=0)
        res["mul_batch"] = bool(np.array_equal(np.asarray(oxy).reshape(-1), r_xy.reshape(-1)) and np.array_equal(oinf, r_inf))
        gxy, ginf = md.mul_by_generator(curve, k)
        r_xy, r_inf = ecref.mul_gen_batch(curve, k, nthreads=B.threads_total)
        res["mul_gen_batch"] = bool(np.array_equal(np.asarray(gxy).reshape(-1), r_xy.reshape(-1)) and np.array_equal(ginf, r_inf))
        lxy, linf = md.lincomb(curve, np.tile(k, 4), np.tile(pxy, 4))          # 20012 terms: bucket method on every device
        r_xy, r_inf = ecref.lincomb(curve, np.tile(k, 4), np.tile(pxy, 4), None, nthreads=B.threads_total)
        res["lincomb"] = bool(np.array_equal(lxy, r_xy) and linf == r_inf)
        bad = k.copy()
        bad[32 * 4999:32 * 5000] = 0xFF
        try:
            md.mul_batch(curve, bad, pxy)
            res["error_index"] = False
        except ecgpu.ScalarRangeError as e:
            res["error_index"] = e.index == 4999
    md.close()
    res["devices"] = B.world
    res["elements"] = n
    return res


def measure_p384(B, steps):
    """Widening record (SURVEY 8(f) rank 4, not a BASELINE config): NIST P-384 variable-base multiplication, 2^18 pairs
    per GPU, through the same kernels with the 12-limb field policy.  Parity: every output against oracle/ecref_p384.c
    (the reference's generic primeorder path over a 384-bit Montgomery field; its duration is the CPU baseline), plus
    the mirror property k*P + (n-k)*P = O on every element and a sample against the big-integer model."""
    import torch

    import pyref

    c = pyref.P384
    eng, host_eng, dev, world, rank = B.eng, B.host_eng, B.dev, B.world, B.rank
    n, nb = 1 << 18, 48
    rng = np.random.default_rng(0xB2000008 + rank)
    K = rng.integers(0, 256, size=(n, nb), dtype=np.uint8)
    K[:, 0] &= 0x7F
    T = rng.integers(0, 256, size=(n, nb), dtype=np.uint8)
    T[:, 0] &= 0x7F
    T[:, nb - 1] |= 1
    pxy, pinf = host_eng.mul_by_generator("p384", T.reshape(-1))
    assert not pinf.any()
    k_host = torch.from_numpy(K.reshape(-1)).pin_memory()
    p_host = torch.from_numpy(np.ascontiguousarray(pxy).reshape(-1)).pin_memory()
    o_host = torch.empty(2 * nb * n, dtype=torch.uint8).pin_memory()
    oi_host = torch.empty(n, dtype=torch.uint8).pin_memory()
    kd, pd = k_host.to(dev), p_host.to(dev)
    oxy = torch.empty(2 * nb * n, dtype=torch.uint8, device=dev)
    oinf = torch.empty(n, dtype=torch.uint8, device=dev)

    def step_dev():
        B.flush.zero_()
        eng.mul_batch_ptr("p384", n, kd.data_ptr(), pd.data_ptr(), 0, oxy.data_ptr(), oinf.data_ptr())

    for _ in range(3):
        step_dev()
    barrier_sync(world)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.timing_enable(True)
    ev0.record()
    for _ in range(steps):
        step_dev()
    ev1.record()
    barrier_sync(world)
    ms = max_over_ranks(ev0.elapsed_time(ev1), world) / steps
    dom_ms, dom_calls = eng.timing_read()
    eng.timing_enable(False)
    host_eng.mul_batch("p384", k_host.numpy(), p_host.numpy(), None, o_host.numpy(), oi_host.numpy())
    barrier_sync(world)
    t0 = time.perf_counter()
    for _ in range(steps):
        host_eng.mul_batch("p384", k_host.numpy(), p_host.numpy(), None, o_host.numpy(), oi_host.numpy())
    barrier_sync(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    # parity: negated scalars give the mirrored points, for every element
    nk = np.frombuffer(b"".join((c.n - int.from_bytes(K[i].tobytes(), "big")).to_bytes(nb, "big") for i in range(n)), np.uint8)
    neg_xy, neg_inf = host_eng.mul_batch("p384", nk, p_host.numpy(), None)
    a, b = o_host.numpy().reshape(n, 2 * nb), np.asarray(neg_xy)
    same_x = bool(np.array_equal(a[:, :nb], b[:, :nb])) and not oi_host.numpy().any() and not neg_inf.any()
    pb = np.frombuffer(c.p.to_bytes(nb, "big"), np.uint8).astype(np.int64)
    # y + y' == p, checked as big-endian byte vectors with carry propagation in numpy (all rows at once)
    sm = a[:, nb:].astype(np.int64) + b[:, nb:].astype(np.int64)
    for j in range(nb - 1, 0, -1):
        sm[:, j - 1] += sm[:, j] >> 8
        sm[:, j] &= 0xFF
    mirrored = bool((sm == pb).all())
    sample_ok = True
    for i in range(0, n, n // 64):
        P = pyref.dec_point(pxy[i].tobytes(), 0, nb)
        sample_ok = sample_ok and pyref.dec_point(a[i].tobytes(), 0, nb) == pyref.mul(c, int.from_bytes(K[i].tobytes(), "big"), P)
    dev_same = bool(np.array_equal(oxy.cpu().numpy(), o_host.numpy()))
    import ecref

    barrier_sync(world)
    t0 = time.perf_counter()
    r_xy, r_inf = ecref.mul_batch("p384", k_host.numpy(), p_host.numpy(), None, nthreads=B.threads)
    cpu_s = time.perf_counter() - t0
    full = bool(np.array_equal(o_host.numpy(), r_xy.reshape(-1)) and np.array_equal(oi_host.numpy(), r_inf))
    cpu_rate = B.sum_over_ranks(n / cpu_s)
    ok = B.all_true(same_x and mirrored and sample_ok and dev_same and full)
    if rank != 0:
        return None
    dom = dom_ms / max(dom_calls, 1)
    imadw = 384 * (4 * 144 + 4 * 144) + 97 * (12 * 144 + 4 * 144)  # 384 dbl (4M+4S) + 97 additions (12M+4S), 144 IMAD.WIDE per 12-limb product
    return {"metric": "scalar-mults/s (p384_varbase)", "value": world * n / (ms * 1e-3), "unit": "scalar-mults/s", "n_gpus": world, "steps": steps,
            "ms_per_step": ms, "config": {"workload": "widening step (SURVEY 8(f) rank 4, not a BASELINE config): NIST P-384 variable base, batch 2^18 per GPU",
                                            "curve": "p384", "batch_per_gpu": n, "record_bytes": {"scalar": 48, "point": 96}},
            "e2e": {"value": world * n * steps / e2e_s, "unit": "scalar-mults/s", "h2d_bytes_per_step": 144 * n, "d2h_bytes_per_step": 97 * n,
                    "matches_device_path": dev_same},
            "bit_exact": ok,
            "bit_exact_coverage": f"every output of every rank vs oracle/ecref_p384.c ({world * n} units); every output: k*P and (n-k)*P mirror each other; "
                                  "64-element sample vs the big-integer model; both oracles are pinned to p384/src/test_vectors/group.rs",
            "roofline_int": {"achieved": imadw * n / (dom * 1e-3), "peak": B.imadw_peak, "frac": imadw * n / (dom * 1e-3) / B.imadw_peak,
                             "unit": "IMAD.WIDE/s (executed)", "imad_wide_per_unit": imadw, "kernel_ms": dom,
                             "note": "12-limb schoolbook product (144 IMAD.WIDE), squarings use the same product; Solinas reduction on the ALU pipe"},
            "cpu_baseline": {"value": cpu_rate, "unit": "scalar-mults/s", "cores": B.cores, "threads": B.threads * world, "kind": "port",
                             "sample": f"the whole workload ({world * n} units), constant-time `*` path (oracle/ecref_p384.c); the same pass is the parity check",
                             "bit_exact_vs_gpu": ok}}


def measure_more_curves(B, steps):
    """Widening record (SURVEY 8(f) rank 4, not a BASELINE config): the other prime-order curves of the reference through
    the same kernels over the generic Montgomery field policy — variable-base multiplication, two kernel waves per GPU and
    curve.  Parity: every output of every rank against oracle/ecref_prime.c (the reference's generic primeorder path:
    RCB formulas for a = -3 / general a, radix-16 constant-time lincomb; its duration is the CPU baseline)."""
    import torch

    import ecref
    import pyref

    eng, host_eng, dev, world, rank = B.eng, B.host_eng, B.dev, B.world, B.rank
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    out = {}
    all_ok = True
    for cid, c in sorted(pyref.EXT_CURVES.items()):
        nb = pyref.fbytes(c)
        nl = (nb + 3) // 4
        # two whole waves of the kernel (128-thread blocks, 4 / 3 / 2 resident per SM by limb count, as ecgpu.cu launches them):
        # every thread runs equally long, so a batch that is not a whole number of waves idles part of the GPU in its last wave
        n = 2 * sms * (2 if nl > 12 else 3 if nl > 8 else 4) * 128
        rng = np.random.default_rng(0xB2000100 + 16 * cid + rank)
        msb = nb - 1 if c.le else 0
        top = c.n >> (8 * (nb - 1))

        def scalars():
            K = rng.integers(0, 256, size=(n, nb), dtype=np.uint8)
            K[:, msb] = K[:, msb] % top
            return K

        K, T = scalars(), scalars()
        T[:, nb - 1 - msb] |= 1                                     # t != 0
        pxy, pinf = host_eng.mul_by_generator(c.name, T.reshape(-1))  # uniformly random points t*G (fixed-base table of the curve)
        assert not pinf.any()
        k_host = torch.from_numpy(K.reshape(-1)).pin_memory()
        p_host = torch.from_numpy(np.ascontiguousarray(pxy).reshape(-1)).pin_memory()
        o_host = torch.empty(2 * nb * n, dtype=torch.uint8).pin_memory()
        oi_host = torch.empty(n, dtype=torch.uint8).pin_memory()
        kd, pd = k_host.to(dev), p_host.to(dev)
        oxy = torch.empty(2 * nb * n, dtype=torch.uint8, device=dev)
        oinf = torch.empty(n, dtype=torch.uint8, device=dev)

        def step_dev():
            B.flush.zero_()
            eng.mul_batch_ptr(c.name, n, kd.data_ptr(), pd.data_ptr(), 0, oxy.data_ptr(), oinf.data_ptr())

        for _ in range(3):
            step_dev()
        barrier_sync(world)
        eng.timing_enable(True)
        for _ in range(steps):
            step_dev()
        torch.cuda.synchronize()
        dom_ms, dom_calls = eng.timing_read()
        eng.timing_enable(False)
        dom = max_over_ranks(dom_ms / max(dom_calls, 1), world)
        host_eng.mul_batch(c.name, k_host.numpy(), p_host.numpy(), None, o_host.numpy(), oi_host.numpy())
        barrier_sync(world)
        t0 = time.perf_counter()
        for _ in range(steps):
            host_eng.mul_batch(c.name, k_host.numpy(), p_host.numpy(), None, o_host.numpy(), oi_host.numpy())
        barrier_sync(world)
        e2e_s = max_over_ranks(time.perf_counter() - t0, world)
        dev_same = bool(np.array_equal(oxy.cpu().numpy(), o_host.numpy()))
        barrier_sync(world)
        t0 = time.perf_counter()
        r_xy, r_inf = ecref.mul_batch(c.name, k_host.numpy(), p_host.numpy(), None, nthreads=B.threads)
        cpu_s = time.perf_counter() - t0
        full = bool(np.array_equal(o_host.numpy(), r_xy.reshape(-1)) and np.array_equal(oi_host.numpy(), r_inf))
        cpu_rate = B.sum_over_ranks(n / cpu_s)
        ok = B.all_true(dev_same and full)
        all_ok = all_ok and ok
        # multiplier slots executed per pair: M = 2 NL^2 + NL (integrated Montgomery product), S = NL(NL+1)/2 + NL^2 + NL;
        # 32 NL doublings (4M+4S; general a: 5M+6S) + 8 NL + 1 Jacobian additions (12M+4S) + table (1 dbl + 1 madd + 6 add)
        M, S = 2 * nl * nl + nl, nl * (nl + 1) // 2 + nl * nl + nl
        if c.p == (1 << c.p.bit_length()) - 1:    # P-521: the Mersenne form of the reduction has no products (FpMontT::redc_mersenne)
            M, S = nl * nl, nl * (nl + 1) // 2
        general_a = (c.a % c.p) != c.p - 3
        dbl = (5 * M + 6 * S) if general_a else (4 * M + 4 * S)
        slots = 32 * nl * dbl + (8 * nl + 1) * (12 * M + 4 * S) + dbl + (8 * M + 3 * S) + 6 * (12 * M + 4 * S)
        out[c.name] = {"value": world * n / (dom * 1e-3), "unit": "scalar-mults/s", "kernel_ms": dom, "record_bytes": nb,
                       "little_endian_records": bool(c.le), "equation_a": "general" if general_a else "-3",
                       "e2e": {"value": world * n * steps / e2e_s, "unit": "scalar-mults/s", "h2d_bytes_per_step": 3 * nb * n,
                               "d2h_bytes_per_step": (2 * nb + 1) * n, "matches_device_path": dev_same},
                       "roofline_int": {"achieved": slots * n / (dom * 1e-3), "peak": B.imadw_peak, "frac": slots * n / (dom * 1e-3) / B.imadw_peak,
                                        "unit": "IMAD.WIDE/s (executed)", "imad_wide_per_unit": slots},
                       "cpu_baseline": {"value": cpu_rate, "unit": "scalar-mults/s", "cores": B.cores, "threads": B.threads * world, "kind": "port",
                                        "sample": f"the whole workload ({world * n} units), constant-time `*` path (oracle/ecref_prime.c)"},
                       "batch_per_gpu": n, "bit_exact": ok}
    if rank != 0:
        return None
    return {"metric": "scalar-mults/s (variable base, per curve)", "unit": "scalar-mults/s", "n_gpus": world, "steps": steps,
            "config": {"workload": "widening step (SURVEY 8(f) rank 4, not a BASELINE config): sm2, brainpoolP256r1/t1, bign-curve256v1, "
                                   "brainpoolP384r1/t1, P-224, P-192, P-521 variable base, two whole kernel waves per GPU and curve (75776 - 113664 "
                                   "pairs on 148 SMs), kernel time by CUDA events (ecg_timing), L2 flushed between steps"},
            "curves": out, "bit_exact": all_ok,
            "bit_exact_coverage": "every output of every rank and curve vs oracle/ecref_prime.c; the oracle is "
                                  "pinned to the reference's p224 / p192 / bignp256 vectors, to the big-integer model and (brainpool, P-224, "
                                  "P-192) to OpenSSL by tests/test_curves_ext.py"}


def measure_consttime_cost(B, steps):
    """What ECG_FLAG_CONSTTIME costs (VERDICT r1 item 8): the variable-base kernels with masked window-table selects and
    branch-free sign folding, k*G through the variable-base routine instead of the fixed-base table; same inputs through a
    default ctx and a constant-time ctx, device-resident, outputs compared byte for byte."""
    import torch

    import ecgpu
    import pyref

    dev, world, rank, host_eng = B.dev, B.world, B.rank, B.host_eng
    ct = ecgpu.Engine([B.local], device_ptrs=True, consttime=True)
    ct.set_stream(torch.cuda.current_stream().cuda_stream)
    out = {}
    all_ok = True
    for name, n in (("k256", 1 << 20), ("p256", 1 << 19)):
        c = pyref.CURVES[name]
        rng = np.random.default_rng(0xB2000200 + rank)
        K = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        K[:, 0] &= 0x7F
        T = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        T[:, 0] &= 0x7F
        T[:, 31] |= 1
        pxy, pinf = host_eng.mul_by_generator(name, T.reshape(-1))
        kd = torch.from_numpy(K.reshape(-1)).to(dev)
        pd = torch.from_numpy(np.ascontiguousarray(pxy).reshape(-1)).to(dev)
        res = {}
        for label, eng in (("vartime", B.eng), ("consttime", ct)):
            oxy = torch.empty(64 * n, dtype=torch.uint8, device=dev)
            oinf = torch.empty(n, dtype=torch.uint8, device=dev)
            gxy = torch.empty(64 * n, dtype=torch.uint8, device=dev)
            ginf = torch.empty(n, dtype=torch.uint8, device=dev)
            times = {}
            for what, call in (("var_base", lambda: eng.mul_batch_ptr(name, n, kd.data_ptr(), pd.data_ptr(), 0, oxy.data_ptr(), oinf.data_ptr())),
                               ("mul_by_generator", lambda: eng.mul_gen_batch_ptr(name, n, kd.data_ptr(), gxy.data_ptr(), ginf.data_ptr()))):
                for _ in range(2):
                    call()
                torch.cuda.synchronize()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for _ in range(steps):
                    B.flush.zero_()
                    call()
                ev1.record()
                torch.cuda.synchronize()
                times[what] = max_over_ranks(ev0.elapsed_time(ev1), world) / steps
            res[label] = (times, oxy, oinf, gxy, ginf)
        same = bool(torch.equal(res["vartime"][1], res["consttime"][1]) and torch.equal(res["vartime"][2], res["consttime"][2])
                    and torch.equal(res["vartime"][3], res["consttime"][3]) and torch.equal(res["vartime"][4], res["consttime"][4]))
        ok = B.all_true(same)
        all_ok = all_ok and ok
        v, t = res["vartime"][0], res["consttime"][0]
        out[name] = {"batch_per_gpu": n,
                     "var_base_ms": {"vartime": v["var_base"], "consttime": t["var_base"], "ratio": t["var_base"] / v["var_base"]},
                     "mul_by_generator_ms": {"vartime_fixed_base_table": v["mul_by_generator"], "consttime_variable_base_routine": t["mul_by_generator"],
                                             "ratio": t["mul_by_generator"] / v["mul_by_generator"]},
                     "consttime_rate": {"var_base": world * n / (t["var_base"] * 1e-3), "mul_by_generator": world * n / (t["mul_by_generator"] * 1e-3),
                                        "unit": "scalar-mults/s"},
                     "bit_exact": ok}
    ct.close()
    if rank != 0:
        return None
    return {"metric": "ms per step (includes the 256 MiB L2 flush write, both arms alike)", "n_gpus": world, "steps": steps,
            "config": {"workload": "cost of ECG_FLAG_CONSTTIME: masked table selects + branch-free sign folding (var-base), variable-base "
                                   "routine instead of the 16-bit fixed-base table (k*G); device-resident operands"},
            "curves": out, "bit_exact": all_ok,
            "bit_exact_coverage": "every output of the constant-time ctx equals the default ctx's (which the other configs compare with the CPU restatement)"}


def measure_hash_to_curve(B, steps):
    """Widening record (SURVEY 8(f) rank 4): RFC 9380 hash_to_curve (RO) over 2^18 messages of 32 bytes per GPU for the two
    SHA-256 suites — SHA-256 expansion, two SSWU maps (one exponentiation each), the isogeny (secp256k1), one addition, batched
    normalisation, all on the device.  Parity: a 256-element sample against the big-integer model (pinned to the reference's
    vectors, tests/test_h2c.py), and every output fed back through ecg_mul_batch with k = 1, whose decoder rejects anything that
    is not a point of the curve."""
    import torch

    import pyref

    eng, host_eng, dev, world, rank = B.eng, B.host_eng, B.dev, B.world, B.rank
    n, mlen = 1 << 18, 32
    dst = b"QUUX-V01-CS02-with-bench"
    out = {}
    all_ok = True
    for name in ("k256", "p256"):
        rng = np.random.default_rng(0xB2000300 + rank)
        M = rng.integers(0, 256, size=(n, mlen), dtype=np.uint8)
        offs = (np.arange(n + 1, dtype=np.uint64) * mlen)
        m_host = torch.from_numpy(M.reshape(-1)).pin_memory()
        o_host = torch.from_numpy(offs.view(np.int64)).pin_memory()
        md, od = m_host.to(dev), o_host.to(dev)
        oxy = torch.empty(64 * n, dtype=torch.uint8, device=dev)
        oinf = torch.empty(n, dtype=torch.uint8, device=dev)
        d = np.frombuffer(dst, np.uint8).copy()
        cid = pyref.CURVE_IDS[name]

        def step_dev():
            B.flush.zero_()
            eng._check(eng.lib.ecg_hash_to_curve_batch(eng._ctx, cid, n, md.data_ptr(), od.data_ptr(), d.ctypes.data, len(dst), 0,
                                                       oxy.data_ptr(), oinf.data_ptr()))

        for _ in range(3):
            step_dev()
        barrier_sync(world)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            step_dev()
        ev1.record()
        barrier_sync(world)
        ms = max_over_ranks(ev0.elapsed_time(ev1), world) / steps
        msgs = [M[i].tobytes() for i in range(n)]
        host_eng.hash_to_curve(name, msgs[:1024], dst)
        m_flat = m_host.numpy()
        barrier_sync(world)
        t0 = time.perf_counter()
        h_xy = h_inf = None
        pin_xy, pin_inf = torch.empty(64 * n, dtype=torch.uint8).pin_memory().numpy(), torch.empty(n, dtype=torch.uint8).pin_memory().numpy()
        for _ in range(steps):
            h_xy, h_inf = host_eng.hash_to_curve_packed(name, m_flat, offs, dst, out_xy=pin_xy, out_inf=pin_inf)      # pinned host buffers: H2D, kernels, D2H
        barrier_sync(world)
        e2e_s = max_over_ranks(time.perf_counter() - t0, world)
        dev_same = bool(np.array_equal(oxy.cpu().numpy(), np.asarray(h_xy).reshape(-1)) and not h_inf.any())
        sample_ok = all(pyref.dec_point(h_xy[i].tobytes(), 0) == pyref.hash_to_curve(name, msgs[i], dst) for i in range(0, n, n // 256))
        ones = np.zeros((n, 32), np.uint8)
        ones[:, 31] = 1
        try:   # every output is a point of the curve: the decoder of ecg_mul_batch accepts all of them, and 1 * P = P
            r_xy, r_inf = host_eng.mul_batch(name, ones.reshape(-1), np.asarray(h_xy).reshape(-1), None)
            on_curve = bool(np.array_equal(r_xy, h_xy) and not r_inf.any())
        except Exception:  # noqa: BLE001
            on_curve = False
        ok = B.all_true(dev_same and sample_ok and on_curve)
        all_ok = all_ok and ok
        out[name] = {"value": world * n / (ms * 1e-3), "unit": "messages/s", "ms_per_step": ms, "messages_per_gpu": n, "message_bytes": mlen,
                     "e2e": {"value": world * n * steps / e2e_s, "unit": "messages/s", "h2d_bytes_per_step": n * (mlen + 8) + 8,
                             "d2h_bytes_per_step": 65 * n, "matches_device_path": dev_same,
                             "note": "host buffers in the C ABI's layout (messages back to back + offsets), copies inside the timed region"},
                     "bit_exact": ok}
    if rank != 0:
        return None
    return {"metric": "messages/s (hash_to_curve, RO)", "unit": "messages/s", "n_gpus": world, "steps": steps,
            "config": {"workload": "widening step (SURVEY 8(f) rank 4): RFC 9380 hash_to_curve, secp256k1_XMD:SHA-256_SSWU_RO_ and "
                                   "P256_XMD:SHA-256_SSWU_RO_, 2^18 messages of 32 bytes per GPU, L2 flushed between steps"},
            "curves": out, "bit_exact": all_ok,
            "bit_exact_coverage": "256-element sample per curve and rank vs the big-integer model (pinned to the reference's RFC 9380 vectors); "
                                  "every output accepted by ecg_mul_batch's on-curve decoder and reproduced by 1 * P; host path == device path"}


def measure_ecdsa_recover(B, steps):
    """Widening record: ECDSA public-key recovery (the Ethereum ecrecover shape) over 2^19 secp256k1 signatures per GPU —
    decompression of R, batched r^-1, u1*G + u2*R, normalisation, all on the device.  Signatures are built so that no host
    inversion is needed: d, k from the seeded hash, R = k*G and Q = d*G on the GPU's fixed-base path, s from the hash too and
    z = s*k - r*d (any 32 bytes are a prehash); low-S normalised with the parity bit flipped, as sign_prehash_recoverable reports it.
    Parity: EVERY recovered key against d*G (itself compared with the CPU restatement in the fixed-base config) and a 128-element
    sample against the big-integer model of recover_from_prehash."""
    import torch

    import pyref

    eng, host_eng, dev, world, rank = B.eng, B.host_eng, B.dev, B.world, B.rank
    c = pyref.K256
    nn = c.n
    n = 1 << 19
    seed = 0xB2000400 + rank
    d = synth_point_scalars("k256", seed, 0, n)
    k = synth_point_scalars("k256", seed ^ 0x5A5A, 0, n)
    sv = synth_point_scalars("k256", seed ^ 0xA5A5, 0, n)
    Qxy, _ = host_eng.mul_by_generator("k256", d)
    Rxy, _ = host_eng.mul_by_generator("k256", k)
    Qxy, Rxy = np.asarray(Qxy).reshape(n, 64), np.asarray(Rxy).reshape(n, 64)
    Z = np.empty((n, 32), np.uint8)
    S = np.empty((n, 64), np.uint8)
    rid = np.empty(n, np.uint8)
    dv, kv, svv = d.reshape(n, 32), k.reshape(n, 32), sv.reshape(n, 32)
    for i in range(n):
        x = int.from_bytes(Rxy[i, :32].tobytes(), "big")
        r = x % nn
        si = int.from_bytes(svv[i].tobytes(), "big")
        z = (si * int.from_bytes(kv[i].tobytes(), "big") - r * int.from_bytes(dv[i].tobytes(), "big")) % nn
        b = (int(Rxy[i, 63]) & 1) | (2 if x >= nn else 0)
        if si > nn // 2:
            si, b = nn - si, b ^ 1
        if r == 0:
            r = 1          # never in practice; keeps the record well-formed (the verdict is then 0 on both sides)
        Z[i] = np.frombuffer(z.to_bytes(32, "big"), np.uint8)
        S[i, :32] = np.frombuffer(r.to_bytes(32, "big"), np.uint8)
        S[i, 32:] = np.frombuffer(si.to_bytes(32, "big"), np.uint8)
        rid[i] = b
    z_host, s_host, r_host = (torch.from_numpy(a.reshape(-1)).pin_memory() for a in (Z, S, rid))
    zd, sd, rd = z_host.to(dev), s_host.to(dev), r_host.to(dev)
    oxy = torch.empty(64 * n, dtype=torch.uint8, device=dev)
    oval = torch.empty(n, dtype=torch.uint8, device=dev)

    def step_dev():
        B.flush.zero_()
        eng._check(eng.lib.ecg_ecdsa_recover_batch(eng._ctx, 0, n, zd.data_ptr(), sd.data_ptr(), rd.data_ptr(), 1, oxy.data_ptr(), oval.data_ptr()))

    for _ in range(3):
        step_dev()
    barrier_sync(world)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step_dev()
    ev1.record()
    barrier_sync(world)
    ms = max_over_ranks(ev0.elapsed_time(ev1), world) / steps
    zn, sn, rn = z_host.numpy(), s_host.numpy(), r_host.numpy()
    host_eng.ecdsa_recover_batch("k256", zn[:32 * 1024], sn[:64 * 1024], rn[:1024], low_s_only=True)
    barrier_sync(world)
    t0 = time.perf_counter()
    h_xy = h_val = None
    pin_xy, pin_val = torch.empty(64 * n, dtype=torch.uint8).pin_memory().numpy(), torch.empty(n, dtype=torch.uint8).pin_memory().numpy()
    for _ in range(steps):
        h_xy, h_val = host_eng.ecdsa_recover_batch("k256", zn, sn, rn, low_s_only=True, out_xy=pin_xy, valid=pin_val)      # pinned host buffers: H2D, kernels, D2H
    barrier_sync(world)
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    dev_same = bool(np.array_equal(oxy.cpu().numpy().reshape(n, 64), h_xy) and np.array_equal(oval.cpu().numpy(), h_val))
    all_keys = bool(h_val.all() and np.array_equal(h_xy, Qxy))
    sample_ok = True
    for i in range(0, n, n // 128):
        q = pyref.ecdsa_recover(c, int.from_bytes(Z[i].tobytes(), "big"), int.from_bytes(S[i, :32].tobytes(), "big"),
                                int.from_bytes(S[i, 32:].tobytes(), "big"), int(rid[i]), True)
        sample_ok = sample_ok and q == (int.from_bytes(h_xy[i, :32].tobytes(), "big"), int.from_bytes(h_xy[i, 32:].tobytes(), "big"))
    ok = B.all_true(dev_same and all_keys and sample_ok)
    if rank != 0:
        return None
    return {"metric": "recoveries/s (ecdsa recover_from_prehash, secp256k1)", "value": world * n / (ms * 1e-3), "unit": "recoveries/s", "n_gpus": world,
            "steps": steps, "ms_per_step": ms, "signatures_per_gpu": n,
            "config": {"workload": "widening step (SURVEY 8(f) ranks 2 + 1 chained): VerifyingKey::recover_from_prehash over 2^19 secp256k1 "
                                   "signatures per GPU (the Ethereum ecrecover shape), low-S enforced, L2 flushed between steps"},
            "e2e": {"value": world * n * steps / e2e_s, "unit": "recoveries/s", "h2d_bytes_per_step": 97 * n, "d2h_bytes_per_step": 65 * n,
                    "matches_device_path": dev_same, "note": "host-buffer C ABI call, pinned host memory, copies inside the timed region"},
            "bit_exact": ok,
            "bit_exact_coverage": "every recovered key == d*G (fixed-base path, itself compared with the CPU restatement in config 4); "
                                  "128-element sample per rank vs the big-integer model of recover_from_prehash (pinned to the reference's vectors)"}


def run_ours(args):
    B = Bench(args)
    world, rank = B.world, B.rank
    line = measure(B, args.workload, args.steps, args.warmup, sample_clocks=True, dump_dir=args.dump_outputs)
    configs = {}
    if args.configs == "all" and args.workload == "k256_varbase":
        sub_steps = min(args.steps, args.sub_steps)
        if rank == 0:
            configs["1_k256_plumbing_cpu"] = config1_plumbing(B)
        for key, wl in (("3_p256_varbase", "p256_varbase"), ("4_k256_fixedbase", "k256_fixedbase"), ("5_k256_lincomb", "k256_lincomb")):
            configs[key] = measure(B, wl, sub_steps, 3, sample_clocks=False)
        configs["6_p384_varbase"] = measure_p384(B, sub_steps)
        configs["7_more_curves"] = measure_more_curves(B, sub_steps)
        configs["8_consttime_cost"] = measure_consttime_cost(B, sub_steps)
        configs["9_hash_to_curve"] = measure_hash_to_curve(B, sub_steps)
        configs["10_k256_schnorr_verify"] = measure(B, "k256_schnorr_verify", sub_steps, 3, sample_clocks=False)
        configs["11_k256_ecdsa_recover"] = measure_ecdsa_recover(B, sub_steps)
        if world > 1:
            configs["strong_scaling"] = strong_scaling(B)
            barrier_sync(world)
            if rank == 0:
                configs["multi_device_parity"] = multi_device_parity(B)
            barrier_sync(world)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        if configs:
            line["configs"] = configs
            line["configs_green"] = bool(all(c.get("bit_exact", True) for c in configs.values() if isinstance(c, dict)))
        print(json.dumps(line), flush=True)


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm (C restatement, oracle/ecref.c — the Rust crate cannot be
    built here: no rustc/cargo, see DESIGN.md) on all host cores; each step = a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import ecref
    import pyref

    curve, op, logn, cfg_idx, unit = WORKLOADS[args.workload]
    seed = SEEDS[args.workload]
    cores, cores_why = host_cores()
    ns = 1 << 16  # units per step
    k = synth_scalars(curve, seed, 0, ns)
    threads = best_thread_count(lambda nt: ecref.mul_gen_batch(curve, k[:32 * 4096], nthreads=nt), cores)
    if op == "schnorr":
        op = "mulgenadd"
    if op != "mulgen":
        t = synth_point_scalars(curve, seed, 0, ns)
        pxy, _ = ecref.mul_gen_batch(curve, t, nthreads=threads)
        pxy = np.ascontiguousarray(pxy).reshape(-1)

    def step():
        if op == "mul":
            ecref.mul_batch(curve, k, pxy, None, nthreads=threads, variant=0)
        elif op == "mulgen":
            ecref.mul_gen_batch(curve, k, nthreads=threads)
        elif op == "mulgenadd":
            ecref.mul_gen_add_batch(curve, k, k, pxy, None, nthreads=threads)
        else:
            ecref.lincomb(curve, k, pxy, None, nthreads=threads)

    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = ns * args.steps / dt
    sample = f"2^16 units per step of the same workload, constant-time `*` path, {threads} threads on {cores} usable cores ({cores_why})"
    line = {
        "impl": "reference",
        "metric": "scalar-mults/sec (var-base, batch) at 1/2/4/8 B200 vs reference Rust CPU" if op == "mul" else f"{unit} ({args.workload})",
        "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1),
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic",
        "config": {"workload": (f"BASELINE.json configs[{cfg_idx}]: " if cfg_idx is not None else "widening step: ") + f"{args.workload}, batch 2^{logn} per GPU",
                   "curve": curve, "step_sample": sample},
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "threads": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40, help="timed steps of the headline workload (and, up to --sub-steps, of every other record)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="k256_varbase", choices=sorted(WORKLOADS))
    ap.add_argument("--log2-batch", type=int, default=0, help="override the per-GPU batch (development only)")
    ap.add_argument("--configs", default="all", choices=["all", "none"],
                    help="all: the headline line also carries a `configs` object with BASELINE.json configs 1, 3, 4, 5 (+ strong scaling at N > 1)")
    ap.add_argument("--sub-steps", type=int, default=10, help="cap on the timed steps of the non-headline configs: they run min(--steps, --sub-steps)")
    ap.add_argument("--strong-log2", type=int, default=23, help="log2 of the strong-scaling batch (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's outputs of its last timed step to DIR/<name>.npy (float32; sampled rows above 2^17)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
