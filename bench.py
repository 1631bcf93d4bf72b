#!/usr/bin/env python3
"""bench.py -- headline benchmark of circl_b200 (contract: see the task statement).

Default workload (BASELINE.json configs[2], the configuration the metric "ML-KEM-768
encaps/sec" is quoted on): 2^20 ML-KEM-768 encapsulations per GPU, every op with
its own 1184-byte encapsulation key (A^T and H(ek) rebuilt on the device per op).
A "step" is one pass of the hot path over that batch.  The same run also measures the
other BASELINE.json configurations and reports them as extra keys of the one JSON line:

  ntt        configs[1]: 2^20-batch Kyber 256-point NTT (forward and inverse)
  keccak     the permutation of the on-device sampler on its own (Keccak-f/s against the ALU-pipe ceiling)
  mldsa65    configs[3]: ML-DSA-65 Sign, 2^18 batch (N = 1)
  mlkem1024  configs[4]: ML-KEM-1024 encaps, 2^21 per GPU (2^24 over 8 GPUs), results gathered to rank 0 (N > 1)

  value     device-resident inputs (HBM), CUDA events, max over ranks
  e2e       the same metric through the C ABI with pinned HOST buffers
            (H2D + kernels + D2H inside the timed region)
  roofline  dominant kernel: algorithmic bytes per launch / its mean launch time
            (CUDA events on the launching stream) vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle (CPU restatement of CIRCL's generic path; Go is not
            available) on a bounded sample of the same inputs, all host threads

--impl reference  times that CPU restatement alone (same metric/config keys).

--steps K sets the number of timed steps of every measurement above.  --dump-outputs DIR writes, after the timed
steps, what the last one returned to its caller (ML-KEM: ct.npy, ss.npy; ML-DSA-65: sig.npy) as float32, one row per
operation, for a fixed seeded sample of the operations whose global indices are in row_index.npy (float64).  The
inputs depend only on the arguments, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree

Q = 3329
WORKLOADS = {
    "mlkem768": dict(k=3, name="ML-KEM-768", ek=1184, ct=1088, bytes_per_op=2336,
                     desc="ML-KEM-768 full encaps (keccakf1600 GenA + NTT matvec) 2^20 batch on 1 B200, per-op ek"),
    "mlkem1024": dict(k=4, name="ML-KEM-1024", ek=1568, ct=1568, bytes_per_op=3200,
                      desc="ML-KEM-1024 encaps 2^24 batch sharded across 8 B200 (2^21 per GPU), per-op ek, per-GPU + aggregate"),
}
MLDSA = dict(name="ML-DSA-65", sk=4032, sig=3309, bytes_per_op=7373,
             desc="ML-DSA-65 Sign 2^18 batch (q=8380417 NTT + rejection loop) on 1 B200, per-op sk, 32-byte messages")
NTT_DESC = "2^20-batch Kyber 256-pt NTT on 1 B200, bit-exact vs common.nttGeneric"
KEY_POOL = ("1024 keys DeriveKeyPair(SHAKE256(0x00||LE32(j))), op i uses key i mod 1024; "
            "m_i = SHAKE256(0x01||LE64(i))")
SM_HZ = 1.965e9
# Keccak-f[1600] on the integer-ALU pipe: 24 rounds x (122 LOP3 + 58 SHF) per state and thread; the pipe issues one
# warp instruction every second clock per SM sub-partition (measured: scripts/ubench_r02.cu reaches 0.496,
# profiles/r02_ubench_keccak.txt), 148 SMs x 4 sub-partitions
KECCAK_INSTR = 24 * 180
KECCAK_PEAK = 148 * 4 * 0.5 * 32 * SM_HZ / KECCAK_INSTR
DUMP_BYTES = 32 << 20  # --dump-outputs: at most this many bytes of float32 output rows


def env_int(name, default):
    return int(os.environ.get(name, default))


def host_threads() -> int:
    """Hardware threads this process may use: CPU affinity, capped by the cgroup CPU quota if one is set."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def ncu_traffic(kernel: str, units_per_launch: float):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json), scaled
    to the units this run's launches process; None if no capture exists for that kernel."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[kernel]
        return t["bytes_per_launch"] * units_per_launch / t["units_per_launch"]
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def dump_rows(total: int, row_bytes: int):
    """Global operation indices --dump-outputs writes: all of them if their rows fit DUMP_BYTES as float32, else a
    fixed seeded sample, sorted."""
    import numpy as np
    k = min(total, DUMP_BYTES // (4 * row_bytes))
    return np.sort(np.random.default_rng(0).choice(total, size=k, replace=False))


def dump_outputs(out_dir: str, rows, arrays: dict):
    """rows: the global indices of the dumped operations; arrays: name -> (len(rows), ...) output rows."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "row_index.npy"), np.asarray(rows, dtype=np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float32))


def mlkem_config(wl, n):
    """The `config` object of an ML-KEM line; identical in our arm and in the reference arm."""
    return {"workload": wl["desc"], "batch_per_gpu": n, "ek": "per-op (stride %d)" % wl["ek"], "key_pool": KEY_POOL,
            "l2": "inputs+outputs %.1f GiB per step, larger than the 126 MB L2" % (n * wl["bytes_per_op"] / 2**30),
            "sharding": "contiguous index ranges per rank; no collective during compute, results gathered to rank 0"}


def mldsa_config(n):
    return {"workload": MLDSA["desc"], "batch_per_gpu": n, "sk": "per-op (stride 4032)",
            "key_pool": "1024 keys DeriveKey(SHAKE256(0x02||LE32(j))), op i uses key i mod 1024; msg_i = SHAKE256(0x03||LE64(i))",
            "l2": "per-op state 65 KB x batch, far larger than L2"}


# ---------------------------------------------------------------- synthetic inputs (SURVEY.md 8(d))
def _shake(tag: int, i: int, width: int, outlen: int) -> bytes:
    import hashlib
    return hashlib.shake_256(bytes([tag]) + i.to_bytes(width, "little")).digest(outlen)


def keygen_seeds(tag: int, count: int, outlen: int):
    """Key-pool seeds: SHAKE256(tag || LE32(j), outlen)  (tag 0x00: ML-KEM d||z, 0x02: ML-DSA xi)."""
    import numpy as np
    return np.frombuffer(b"".join(_shake(tag, j, 4, outlen) for j in range(count)), dtype=np.uint8).reshape(count, outlen)


def op_seeds(tag: int, first: int, n: int):
    """Per-op 32-byte inputs: SHAKE256(tag || LE64(i), 32)  (tag 0x01: ML-KEM m_i, 0x03: ML-DSA msg_i)."""
    import numpy as np
    return np.frombuffer(b"".join(_shake(tag, i, 8, 32) for i in range(first, first + n)), dtype=np.uint8).reshape(n, 32)


def mlkem_key_pool(k: int, count: int, on_gpu: bool):
    """1024 real encapsulation keys DeriveKeyPair(SHAKE256(0x00 || LE32(j), 64)).  Our arm derives them with the
    GPU KeyGen of this library (the product path); the reference arm with the CPU restatement."""
    import numpy as np
    seeds = keygen_seeds(0x00, count, 64)
    if on_gpu:
        from circl_b200 import mlkem
        name = {2: "ML-KEM-512", 3: "ML-KEM-768", 4: "ML-KEM-1024"}[k]
        return mlkem.ByName(name).DeriveKeyPairBatch(seeds)[0]
    import oracle
    return np.stack([np.frombuffer(oracle.mlkem_keygen(k, s.tobytes())[0], dtype=np.uint8) for s in seeds])


def mldsa_key_pool(count: int, on_gpu: bool):
    """1024 real ML-DSA-65 private keys DeriveKey(SHAKE256(0x02 || LE32(j), 32))."""
    import numpy as np
    seeds = keygen_seeds(0x02, count, 32)
    if on_gpu:
        from circl_b200 import mldsa
        return mldsa.ByName("ML-DSA-65").DeriveKeyBatch(seeds)[1]
    import oracle
    return np.stack([np.frombuffer(oracle.mldsa65_keygen(s.tobytes())[1], dtype=np.uint8) for s in seeds])


def synth_polys(first_poly: int, n: int, device="cpu"):
    """c = (splitmix64(0x243F6A8885A308D3 + idx) mod 6658) - 3329, idx = poly*256 + j: the RandAbsLeQ
    distribution of pke/kyber/internal/common/ntt_test.go:41-47 from a counter-based generator.
    Returns an (n, 256) int16 torch tensor on `device` (two's-complement int64 arithmetic, chunked)."""
    import torch

    def s64(x):  # uint64 constant -> the int64 with the same bits
        return x - (1 << 64) if x >= (1 << 63) else x

    def lsr(z, k):  # logical shift right on int64 bit patterns
        return (z >> k) & ((1 << (64 - k)) - 1)

    out = torch.empty((n, 256), dtype=torch.int16, device=device)
    chunk = 1 << 17
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        idx = torch.arange((first_poly + lo) * 256, (first_poly + lo + m) * 256, dtype=torch.int64, device=device)
        z = idx + s64((0x243F6A8885A308D3 + 0x9E3779B97F4A7C15) & ((1 << 64) - 1))
        z = (z ^ lsr(z, 30)) * s64(0xBF58476D1CE4E5B9)
        z = (z ^ lsr(z, 27)) * s64(0x94D049BB133111EB)
        z = z ^ lsr(z, 31)
        r = torch.remainder(z, 6658) + torch.where(z < 0, (1 << 64) % 6658, 0)
        out[lo:lo + m] = (torch.remainder(r, 6658) - 3329).to(torch.int16).view(m, 256)
    return out


# ---------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  The region is short (5 steps of ~18 ms), so the samples
    come from NVML in a thread (one query ~ 0.1 ms, every 2 ms) -- the same counters `nvidia-smi --query-gpu=clocks.sm,
    clocks.max.sm,clocks_event_reasons.*` prints (B200_PROFILING.md), which is the fallback when pynvml is missing:
    nvidia-smi itself needs longer to start than the region lasts."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.handle, self.thread, self.stop_flag, self.samples, self.mask, self.max_mhz = None, None, None, False, [], 0, None
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes the visible devices; map through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            ids = [x.strip() for x in vis.split(",")] if vis else []
            if index < len(ids) and ids[index].startswith("GPU-"):
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(ids[index])
            else:
                phys = int(ids[index]) if index < len(ids) and ids[index].isdigit() else index
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml is not None:
            self.stop_flag, self.samples, self.mask = False, [], 0
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            sm = self.samples
            load = [x for x in sm if x >= 0.5 * max(sm)] if sm else []
            return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(name for name, bit in self.REASONS if self.mask & bit), "samples": len(sm),
                    "source": "nvml, every 2 ms during the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        # "under load" = samples in the upper half of what was seen (idle samples bracket the region)
        load = [x for x in sm if x >= 0.5 * max(sm)] if sm else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ---------------------------------------------------------------- reference arm (CPU restatement)
def config1_cpu(threads: int):
    """BASELINE.json configs[0]: ML-KEM-768 Encapsulate, 1024-op loop on the CPU path with the keys and seeds of the
    KAT procedure (kem/kyber/kat_test.go:48-81 extended from 100 to 1024 counts): DRBG seed = bytes 0..47; per count
    seed <- DRBG(48), g2 = DRBG(seed), kseed <- g2(64), eseed <- g2(32).  Timed with the key already unmarshalled (as
    in the reference's BenchmarkEncapsulate) and including UnmarshalBinaryPublicKey, on one thread and on all."""
    import numpy as np
    import oracle
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from nist_drbg import DRBG
    g = DRBG(bytes(range(48)))
    eks, ms = [], []
    for _ in range(1024):
        g2 = DRBG(g.fill(48))
        kseed, eseed = g2.fill(64), g2.fill(32)
        eks.append(np.frombuffer(oracle.mlkem_keygen(3, kseed)[0], dtype=np.uint8))
        ms.append(np.frombuffer(eseed, dtype=np.uint8))
    eks, ms = np.stack(eks), np.stack(ms)
    parsed = oracle.mlkem_parse_keys(3, eks)
    out = {"ops": 1024, "inputs": "kem/kyber/kat_test.go:48-81 DRBG procedure, counts 0..1023", "unit": "encaps/s",
           "arm": "generic restatement (oracle/kyber.c); including_unmarshal_avx2 = the same loop on the AVX2 arm"}
    ref = None
    for label, nt in (("1_thread", 1), ("all_threads", threads)):
        best_p = best_u = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            ct, ss = oracle.mlkem_encaps_parsed_batch(3, parsed, ms, nthreads=nt)
            best_p = min(best_p, time.perf_counter() - t0)
            t0 = time.perf_counter()
            ct2, ss2, fails = oracle.mlkem_encaps_batch(3, eks, ms, nthreads=nt)
            best_u = min(best_u, time.perf_counter() - t0)
            assert fails == 0 and np.array_equal(ct, ct2) and np.array_equal(ss, ss2)
        ref = (ct, ss)
        best_a = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            ct3, ss3, fails = oracle.mlkem_encaps_batch_avx2(3, eks, ms, nthreads=nt)
            best_a = min(best_a, time.perf_counter() - t0)
            assert fails == 0 and np.array_equal(ct, ct3) and np.array_equal(ss, ss3)
        out[label] = {"cores": nt, "pk_pre_parsed": 1024 / best_p, "including_unmarshal": 1024 / best_u,
                      "including_unmarshal_avx2": 1024 / best_a}
    return out, eks, ms, ref


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    import numpy as np
    import oracle
    threads = host_threads()
    wl = WORKLOADS[args.workload]
    n = 1 << args.batch_log2
    sample = min(n, 1 << 17)
    keys = mlkem_key_pool(wl["k"], 1024, on_gpu=False)
    idx = np.arange(sample) % 1024
    eks = np.ascontiguousarray(keys[idx])
    seeds = op_seeds(0x01, 0, sample)
    # Two CPU arms (both C restatements; CIRCL itself is Go and cannot be built here):
    #   avx2     oracle/kyber_avx2.c  -- CIRCL's real amd64 path: f1600x4AVX2 for matrix A, nttAVX2 / invNttAVX2 / mulHatAVX2
    #   generic  oracle/kyber.c       -- CIRCL's purego path
    # The line's `value` (the denominator of the driver's ratio) is the FASTER, AVX2 one.
    arms = {}
    for arm, fn in (("avx2", oracle.mlkem_encaps_batch_avx2), ("generic", oracle.mlkem_encaps_batch)):
        times = []
        for step in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            _, _, fails = fn(wl["k"], eks, seeds, nthreads=threads)
            dt = time.perf_counter() - t0
            assert fails == 0
            if step >= args.warmup:
                times.append(dt)
        t0 = time.perf_counter()
        fn(wl["k"], eks[:1 << 13], seeds[:1 << 13], nthreads=1)
        arms[arm] = {"ms": 1e3 * sum(times) / len(times), "single_thread": (1 << 13) / (time.perf_counter() - t0)}
    ms = arms["avx2"]["ms"]
    value = sample / (ms * 1e-3)
    one = arms["avx2"]["single_thread"]
    c1, _, _, _ = config1_cpu(threads) if wl["k"] == 3 else (None, None, None, None)
    line = {
        "impl": "reference", "metric": f"{wl['name']} encaps/sec", "value": value, "unit": "encaps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": "synthetic",
        "config": mlkem_config(wl, n),
        "cpu_baseline": {"value": value, "unit": "encaps/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} ops per step (first 2^17 of the batch) incl. per-op key parse; C restatement "
                                   "of CIRCL's amd64 fast path (4-way AVX2 Keccak for matrix A, 16-lane AVX2 NTT / InvNTT / "
                                   "MulHat; oracle/kyber_avx2.c); CIRCL itself is Go and no Go toolchain exists here",
                         "single_thread": one,
                         "generic": {"value": sample / (arms["generic"]["ms"] * 1e-3),
                                     "single_thread": arms["generic"]["single_thread"],
                                     "what": "C restatement of CIRCL's purego path (oracle/kyber.c), same sample and threads"},
                         "config1": c1},
        "e2e": {"value": value, "unit": "encaps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_reference_mldsa(args):
    import numpy as np
    import oracle
    if env_int("RANK", 0) != 0:
        return 0
    threads = host_threads()
    n = 1 << (args.batch_log2 if args.batch_log2 != 20 else 18)
    sample = 1 << 12
    keys = mldsa_key_pool(1024, on_gpu=False)
    sks = np.ascontiguousarray(keys[np.arange(sample) % 1024])
    msgs = [bytes(m) for m in op_seeds(0x03, 0, sample)]
    times = []
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        oracle.mldsa65_sign_batch(sks, msgs, nthreads=threads)
        if step >= args.warmup:
            times.append(time.perf_counter() - t0)
    ms = 1e3 * sum(times) / len(times)
    v = sample / (ms * 1e-3)
    print(json.dumps({
        "impl": "reference", "metric": "ML-DSA-65 sign/sec", "value": v, "unit": "sign/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "uint32", "data": "synthetic", "config": mldsa_config(n),
        "cpu_baseline": {"value": v, "unit": "sign/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} signatures per step, per-op sk expansion, C restatement of CIRCL's generic path"},
        "e2e": {"value": v, "unit": "sign/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
    return 0


# ---------------------------------------------------------------- shared run context
class Ctx:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.args = args
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        import circl_b200
        from circl_b200._ffi import lib, check
        self.cb, self.L, self.check = circl_b200, lib(), check
        # NUMA first: this thread (and the pinned buffers it allocates from now on) stays next to its GPU
        self.numa_cpus = self.L.cb200_bind_thread_to_device(self.local)
        torch.cuda.set_device(self.local)
        self.dist = dist
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        circl_b200.init(self.local)
        self.peak, self.peak_kind = measured_peak()
        self.torch = torch

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def profile(self, fn, reps=1):
        """Per-kernel-class CUDA-event timing of fn() (serialised on one stream inside the library)."""
        L, check = self.L, self.check
        check(L.cb200_profile_enable(1))
        for _ in range(reps):
            fn()
        nk = L.cb200_profile_kernel_count()
        ms_tot = (ctypes.c_double * nk)()
        cnt = (ctypes.c_uint64 * nk)()
        check(L.cb200_profile_read(ms_tot, cnt, nk))
        check(L.cb200_profile_enable(0))
        return {L.cb200_profile_kernel_name(i).decode(): {"ms_total": ms_tot[i] / reps, "launches": int(cnt[i]) // reps}
                for i in range(nk) if cnt[i]}


# ---------------------------------------------------------------- ML-KEM encaps (configs 3 and 5)
def bench_mlkem(cx: Ctx, wl_key: str, log2n: int, steps: int, warmup: int, with_profile=True, with_cpu=True,
                e2e_steps=5, sampler=None, dump_dir=None):
    import numpy as np
    torch, L, check = cx.torch, cx.L, cx.check
    from circl_b200 import mlkem
    wl = WORKLOADS[wl_key]
    scheme = mlkem.ByName(wl["name"])
    n = 1 << log2n
    rank, world = cx.rank, cx.world

    # ---- inputs: shard r owns global op indices [r*n, (r+1)*n); op i uses key pool[i mod 1024]
    keys = mlkem_key_pool(wl["k"], 1024, on_gpu=True)
    gidx = (np.arange(n, dtype=np.int64) + rank * n) % 1024
    eks_h = torch.empty((n, wl["ek"]), dtype=torch.uint8, pin_memory=True)
    eks_h.numpy()[:] = keys[gidx]
    seeds_h = torch.empty((n, 32), dtype=torch.uint8, pin_memory=True)
    seeds_h.numpy()[:] = op_seeds(0x01, rank * n, n)
    ct_h = torch.empty((n, wl["ct"]), dtype=torch.uint8, pin_memory=True)
    ss_h = torch.empty((n, 32), dtype=torch.uint8, pin_memory=True)
    eks_d, seeds_d = eks_h.cuda(), seeds_h.cuda()
    ct_d = torch.empty((n, wl["ct"]), dtype=torch.uint8, device="cuda")
    ss_d = torch.empty((n, 32), dtype=torch.uint8, device="cuda")

    # N > 1: results are gathered to rank 0 in global index order (the one exchange of this path).  The flow pushes every
    # sub-batch of 8192 results into rank 0's buffer as soon as it exists (cb200_mlkem_encaps_push: peer copies by the
    # copy engines over NVLink) while the next sub-batches compute.
    from circl_b200.shard import RowGather
    pg = RowGather(n, [wl["ct"], 32], transport="ipc") if world > 1 else None

    def step_device(do_gather=True):
        push = (pg.dst_ptr(0), pg.dst_ptr(1)) if (pg is not None and do_gather) else None
        scheme.EncapsulateBatch(eks_d, seeds_d, ct=ct_d, ss=ss_d, push=push)

    def step_host():
        check(L.cb200_mlkem_encaps(wl["k"], eks_h.data_ptr(), wl["ek"], seeds_h.data_ptr(), ct_h.data_ptr(),
                                   ss_h.data_ptr(), None, n))

    # ---- device-resident timing (inputs + outputs per step far larger than the 126 MB L2)
    for _ in range(warmup):
        step_device()
    cx.barrier()
    if sampler is not None and rank == 0:
        sampler.start()
    launches0 = cx.cb.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step_device()
    ev1.record()
    cx.barrier()
    launches = cx.cb.launch_count() - launches0
    ms_step = cx.max_over_ranks(ev0.elapsed_time(ev1) / steps)
    scheme.check_last_status()
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    if dump_dir is not None and rank == 0:
        # N > 1: the caller of the gathered path receives every rank's rows in rank 0's buffer
        ct_all, ss_all = (pg.matrix(0), pg.matrix(1)) if pg is not None else (ct_d, ss_d)
        rows = dump_rows(world * n, wl["ct"] + 32)
        sel = torch.as_tensor(rows, device=ct_all.device)
        dump_outputs(dump_dir, rows, {"ct": ct_all[sel].cpu().numpy(), "ss": ss_all[sel].cpu().numpy()})

    # ---- N > 1: parity of the GATHERED buffer, the same step without the gather, and the gather alone
    gather = None
    if world > 1:
        match = None
        if rank == 0:
            import oracle
            rng = np.random.default_rng(2024)
            idx = sorted(set([0, world * n - 1] + [r * n + int(x) for r in range(world)
                                                    for x in list(rng.integers(0, n, size=14)) + [0, n - 1]]))
            sel = torch.as_tensor(idx, device="cuda")
            got_ct, got_ss = pg.matrix(0)[sel].cpu().numpy(), pg.matrix(1)[sel].cpu().numpy()
            match = True
            for j, i in enumerate(idx):
                wct, wss = oracle.mlkem_encaps(wl["k"], keys[i % 1024].tobytes(), op_seeds(0x01, i, 1)[0].tobytes())
                match &= got_ct[j].tobytes() == wct and got_ss[j].tobytes() == wss
            match = bool(match)
        cx.barrier()
        ev0.record()
        for _ in range(steps):
            step_device(do_gather=False)
        ev1.record()
        cx.barrier()
        ms_nogather = cx.max_over_ranks(ev0.elapsed_time(ev1) / steps)
        ev0.record()
        pg.push([ct_d, ss_d], 0, n)
        pg.flush(ct_d)
        ev1.record()
        cx.barrier()
        ms_gather = cx.max_over_ranks(ev0.elapsed_time(ev1))
        nbytes = (world - 1) * n * (wl["ct"] + 32)
        gather = {"to": "rank 0", "bytes_per_step": nbytes, "chunks": (n + 8191) // 8192, "ms_alone": ms_gather,
                  "rank0_ingress_GBps": nbytes / 1e9 / (ms_gather * 1e-3),
                  "ms_per_step_without_gather": ms_nogather, "exposed_ms": ms_step - ms_nogather,
                  "gathered_outputs_match": match, "checked_rows": (len(idx) if rank == 0 else None),
                  "transport": "CUDA IPC mapping of rank 0's buffer + cudaMemcpyAsync peer copies on a copy stream "
                               "(copy engines over NVLink; no SM), issued by the encaps flow itself per sub-batch of 8192 "
                               "results (cb200_mlkem_encaps_push); torch.distributed/NCCL only for the handle and barriers",
                  "note": "value includes the gather, overlapped sub-batch by sub-batch with the kernels; the strided "
                          "sample of the gathered buffer on rank 0 is compared with the oracle"}

    # ---- end to end through the C ABI with pinned host buffers
    e2e = None
    if e2e_steps:
        for _ in range(2):
            step_host()
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_host()
        torch.cuda.synchronize()
        e2e_ms = cx.max_over_ranks(1e3 * (time.perf_counter() - t0) / e2e_steps)
        cx.barrier()
        same = bool(torch.equal(ct_h[: 1 << 12], ct_d[: 1 << 12].cpu()) and torch.equal(ss_h[: 1 << 12], ss_d[: 1 << 12].cpu()))
        e2e = {"value": world * n / (e2e_ms * 1e-3), "unit": "encaps/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": n * (wl["ek"] + 32), "d2h_bytes_per_step": n * (wl["ct"] + 32 + 1),
               "host_vs_device_outputs_equal": same,
               "numa": "rank thread and its pinned buffers bound to the %d CPUs next to its GPU" % cx.numa_cpus
                       if cx.numa_cpus else "topology unknown, unbound"}
        # The floor of that number on this box: the same bytes of the same pinned buffers, copied in and out at the same
        # time on two streams by every rank at once, and no kernel at all.
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

        def copies_only():
            with torch.cuda.stream(s_in):
                eks_d.copy_(eks_h, non_blocking=True)
                seeds_d.copy_(seeds_h, non_blocking=True)
            with torch.cuda.stream(s_out):
                ct_h.copy_(ct_d, non_blocking=True)
                ss_h.copy_(ss_d, non_blocking=True)
        copies_only()
        torch.cuda.synchronize()
        cx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            copies_only()
        torch.cuda.synchronize()
        copy_ms = cx.max_over_ranks(1e3 * (time.perf_counter() - t0) / e2e_steps)
        cx.barrier()
        e2e["copies_only_ms_per_step"] = copy_ms
        e2e["copies_only_GBps_per_direction_all_ranks"] = world * n * (wl["ek"] + 32) / (copy_ms * 1e6)
        e2e["share_of_copy_floor"] = copy_ms / e2e_ms

    # ---- per-kernel event timing (separate pass, not part of `value`)
    roofline = None
    if with_profile:
        kernels = cx.profile(lambda: scheme.EncapsulateBatch(eks_d, seeds_d, ct=ct_d, ss=ss_d), reps=2)
        total_kernel_ms = sum(v["ms_total"] for v in kernels.values())
        dom_name = max(kernels, key=lambda k_: kernels[k_]["ms_total"])
        dom = kernels[dom_name]
        units_per_launch = n / dom["launches"]
        dom_ms = dom["ms_total"] / dom["launches"]
        achieved = wl["bytes_per_op"] * units_per_launch / (dom_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": cx.peak, "unit": "GB/s",
                    "frac": achieved / cx.peak, "traffic": ncu_traffic(dom_name, units_per_launch),
                    "peak_kind": cx.peak_kind, "share_of_step": dom["ms_total"] / total_kernel_ms,
                    "note": "path is integer-ALU (Keccak) bound, not HBM bound; achieved = %d algorithmic B/op x %d ops per "
                            "launch / mean launch time; traffic = ncu dram bytes per launch.  kernels_ms_per_step comes from "
                            "a profiling pass that serialises the two internal lanes on one stream, so it sums to more "
                            "than ms_per_step; share_of_step is a share of that sum" % (wl["bytes_per_op"], int(units_per_launch)),
                    "kernels_ms_per_step": {k_: round(v["ms_total"], 4) for k_, v in kernels.items()}}
        # The binding resource is the integer-ALU pipe, so state that roofline too (Keccak-f/s of the kernel against the
        # measured ceiling of the permutation, see KECCAK_PEAK)
        k = wl["k"]
        perms = {"mlkem_sample": 3 * k * k + (2 * k + 1), "mlkem_hash_ek": (384 * k + 32) // 136 + 1}.get(dom_name)
        if perms:
            alu_ach = perms * units_per_launch / (dom_ms * 1e-3)
            roofline["alu"] = {"bound": "int-alu", "achieved": alu_ach, "peak": KECCAK_PEAK, "unit": "keccak-f/s",
                               "frac": alu_ach / KECCAK_PEAK,
                               "note": "%d Keccak-f per op in this kernel (3 SHAKE128 blocks per matrix entry + 1 SHAKE256 "
                                       "block per noise polynomial) x 180 ALU-pipe instructions per round; the remainder "
                                       "of the pipe time is rejection parsing and CBD" % perms}

    # ---- CPU baseline (rank 0, N = 1 only): oracle port on a bounded sample, outputs cross-checked
    cpu = None
    if with_cpu and rank == 0 and world == 1:
        import oracle
        threads = host_threads()
        sample = min(n, 1 << 17)
        eks_s = np.ascontiguousarray(eks_h.numpy()[:sample])
        seeds_s = np.ascontiguousarray(seeds_h.numpy()[:sample])
        oracle.mlkem_encaps_batch(wl["k"], eks_s[:1024], seeds_s[:1024], nthreads=threads)
        t0 = time.perf_counter()
        wct, wss, fails = oracle.mlkem_encaps_batch(wl["k"], eks_s, seeds_s, nthreads=threads)
        dt = time.perf_counter() - t0
        parity = bool(fails == 0 and np.array_equal(wct, ct_h.numpy()[:sample]) and np.array_equal(wss, ss_h.numpy()[:sample]))
        t0 = time.perf_counter()
        oracle.mlkem_encaps_batch(wl["k"], eks_s[:1 << 13], seeds_s[:1 << 13], nthreads=1)
        one = (1 << 13) / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        act, ass, af = oracle.mlkem_encaps_batch_avx2(wl["k"], eks_s, seeds_s, nthreads=threads)
        adt = time.perf_counter() - t0
        parity &= bool(af == 0 and np.array_equal(act, wct) and np.array_equal(ass, wss))
        t0 = time.perf_counter()
        oracle.mlkem_encaps_batch_avx2(wl["k"], eks_s[:1 << 13], seeds_s[:1 << 13], nthreads=1)
        aone = (1 << 13) / (time.perf_counter() - t0)
        cpu = {"value": sample / adt, "unit": "encaps/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} ops of the batch, all {threads} host threads; C restatement of CIRCL's amd64 fast "
                         "path (AVX2: 4-way Keccak for matrix A, 16-lane NTT / InvNTT / MulHat; oracle/kyber_avx2.c) -- "
                         "no Go toolchain on this image",
               "outputs_match_gpu": parity, "single_thread": aone,
               "generic": {"value": sample / dt, "single_thread": one,
                           "what": "C restatement of CIRCL's purego path (oracle/kyber.c), same sample and threads"}}
        if wl["k"] == 3:
            # BASELINE configs[0] beside it, and the same 1024 KAT operations through the GPU path
            c1, keks, kms, (kct, kss) = config1_cpu(threads)
            gct, gss = scheme.EncapsulateBatch(keks, kms)
            c1["gpu_outputs_match"] = bool(np.array_equal(gct, kct) and np.array_equal(gss, kss))
            cpu["config1"] = c1
    if pg is not None:
        cx.barrier()
        pg.close()
    rec = {"metric": f"{wl['name']} encaps/sec", "value": world * n / (ms_step * 1e-3), "unit": "encaps/s",
           "per_gpu": n / (ms_step * 1e-3), "ms_per_step": ms_step, "config": mlkem_config(wl, n), "e2e": e2e,
           "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "gather": gather}
    del eks_d, seeds_d, ct_d, ss_d, eks_h, ct_h
    torch.cuda.empty_cache()
    return rec, clocks


# ---------------------------------------------------------------- raw NTT (config 2) and the Keccak permutation
def bench_ntt(cx: Ctx, steps: int, warmup: int, with_cpu: bool):
    torch, L, check = cx.torch, cx.L, cx.check
    from circl_b200 import kyber
    npoly = 1 << 20
    polys_d = synth_polys(cx.rank * npoly, npoly, device="cuda")
    polys_h = torch.empty((npoly, 256), dtype=torch.int16, pin_memory=True)
    polys_h.copy_(polys_d)
    # The transforms run in place, so every call gets a fresh copy of the batch: |c| <= q, the input contract of
    # nttGeneric / invNTTGeneric (ntt.go:60-66, 145-150) and the distribution of the reference's own test
    # (RandAbsLeQ, ntt_test.go:41-47).  The copy and an L2 flush sit outside the event-timed call.  A second figure
    # times the same kernels on arbitrary int16 inputs, which take the general (int16 wrap-around exact) path.
    pristine = polys_d.clone()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    any16 = None
    ntt = {}

    def timed(fn, src, reps):
        ts = []
        for i in range(warmup + reps):
            polys_d.copy_(src)
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn(polys_d)
            b.record()
            if i >= warmup:
                ts.append((a, b))
        cx.barrier()
        return cx.max_over_ranks(statistics.median(a.elapsed_time(b) for a, b in ts))

    for label, fn in (("forward", kyber.ntt_), ("inverse", kyber.inv_ntt_)):
        ms = timed(fn, pristine, steps)
        gbs = npoly * 1024 / (ms * 1e-3) / 1e9
        ntt[label] = {"value": cx.world * npoly / (ms * 1e-3), "unit": "NTT/s", "ms_per_step": ms,
                      "roofline": {"bound": "hbm", "achieved": gbs, "peak": cx.peak, "unit": "GB/s",
                                   "frac": gbs / cx.peak, "peak_kind": cx.peak_kind,
                                   "traffic": ncu_traffic("kyber_ntt" if label == "forward" else "kyber_invntt", npoly)}}
        if any16 is None:
            g = torch.Generator(device="cuda").manual_seed(1 + cx.rank)
            any16 = torch.randint(-32768, 32768, (npoly, 256), device="cuda", dtype=torch.int32, generator=g).to(torch.int16)
        ms_any = timed(fn, any16, steps)
        ntt[label]["any_int16_inputs"] = {"ms_per_step": ms_any, "value": cx.world * npoly / (ms_any * 1e-3),
                                          "frac": npoly * 1024 / (ms_any * 1e-3) / 1e9 / cx.peak}
    del pristine, flush, any16
    ntt["config"] = {"workload": NTT_DESC, "polys_per_gpu": npoly, "bytes_per_ntt": 1024,
                     "inputs": "RandAbsLeQ (|c| <= q) restored before every timed call; any_int16_inputs: uniform int16",
                     "l2": "input 512 MiB > 126 MB L2, flushed by a 256 MiB write before every timed call; "
                           "kernel reads and writes every byte once"}
    host_src = polys_h.clone()
    e2e_s = []
    for i in range(warmup + steps):
        polys_h.copy_(host_src)
        t0 = time.perf_counter()
        check(L.cb200_kyber_ntt(polys_h.data_ptr(), npoly, 0))
        if i >= warmup:
            e2e_s.append(time.perf_counter() - t0)
    del host_src
    ntt["e2e"] = {"value": cx.world * npoly / (sum(e2e_s) / len(e2e_s)), "unit": "NTT/s",
                  "h2d_bytes_per_step": npoly * 512, "d2h_bytes_per_step": npoly * 512}
    if with_cpu and cx.rank == 0 and cx.world == 1:
        import oracle
        threads = host_threads()
        ps = synth_polys(0, 1 << 16).numpy()
        t0 = time.perf_counter()
        oracle.kyber_ntt_inplace_mt(ps, False, threads)
        ntt["cpu_baseline"] = {"value": (1 << 16) / (time.perf_counter() - t0), "unit": "NTT/s", "cores": threads,
                               "kind": "port", "sample": "2^16 polynomials, nttGeneric restatement"}
    del polys_d, polys_h
    torch.cuda.empty_cache()
    return ntt


def bench_keccak(cx: Ctx, steps: int, warmup: int):
    """cb200_keccak_f1600 on 2^22 device-resident states (800 MiB): the permutation of the on-device sampler alone."""
    torch = cx.torch
    from circl_b200 import keccak
    n = 1 << 22
    st = torch.arange(n * 25, dtype=torch.int64, device="cuda").view(n, 25)
    for _ in range(warmup):
        keccak.permute_(st)
    cx.barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in evs:
        a.record()
        keccak.permute_(st)
        b.record()
    cx.barrier()
    ms = cx.max_over_ranks(statistics.median(a.elapsed_time(b) for a, b in evs))
    v = n / (ms * 1e-3)
    gbs = n * 400 / (ms * 1e-3) / 1e9
    del st
    torch.cuda.empty_cache()
    return {"metric": "Keccak-f[1600]/sec", "value": cx.world * v, "unit": "keccak-f/s", "ms_per_step": ms,
            "config": {"workload": "cb200_keccak_f1600 on 2^22 states per GPU (200 B each, in place), 24 rounds",
                       "l2": "800 MiB per pass, larger than L2"},
            "roofline": {"bound": "int-alu", "achieved": v, "peak": KECCAK_PEAK, "unit": "keccak-f/s", "frac": v / KECCAK_PEAK,
                         "note": "peak = 148 SMs x 4 sub-partitions x 0.5 warp-instr/clk x 32 lanes x 1.965 GHz / (24 x 180 "
                                 "LOP3+SHF); scripts/ubench_r02.cu measures 4.27e9/s for the bare register loop",
                         "hbm": {"achieved": gbs, "peak": cx.peak, "unit": "GB/s", "frac": gbs / cx.peak}}}


# ---------------------------------------------------------------- ML-DSA-65 (BASELINE configs[3])
def bench_mldsa(cx: Ctx, log2n: int, steps: int, warmup: int, with_cpu: bool, sampler=None, dump_dir=None):
    import numpy as np
    torch, L, check = cx.torch, cx.L, cx.check
    rank, world = cx.rank, cx.world
    n = 1 << log2n
    keys = mldsa_key_pool(1024, on_gpu=True)
    gidx = (np.arange(n, dtype=np.int64) + rank * n) % 1024
    sk_h = torch.empty((n, 4032), dtype=torch.uint8, pin_memory=True)
    sk_h.numpy()[:] = keys[gidx]
    msg_h = torch.empty((n, 32), dtype=torch.uint8, pin_memory=True)
    msg_h.numpy()[:] = op_seeds(0x03, rank * n, n)
    off_h = torch.arange(0, 32 * (n + 1), 32, dtype=torch.int64).pin_memory()
    sig_h = torch.empty((n, 3309), dtype=torch.uint8, pin_memory=True)
    sk_d, msg_d, off_d = sk_h.cuda(), msg_h.cuda(), off_h.cuda()
    sig_d = torch.empty((n, 3309), dtype=torch.uint8, device="cuda")
    st_d = torch.zeros((n,), dtype=torch.uint8, device="cuda")
    attempts = ctypes.c_uint64(0)

    def step_device():
        check(L.cb200_set_stream(torch.cuda.current_stream().cuda_stream))
        check(L.cb200_mldsa65_sign(sk_d.data_ptr(), 4032, msg_d.data_ptr(), off_d.data_ptr(), None, 0, None,
                                   sig_d.data_ptr(), st_d.data_ptr(), n, 0, ctypes.cast(ctypes.pointer(attempts), ctypes.c_void_p)))

    def step_host():
        check(L.cb200_mldsa65_sign(sk_h.data_ptr(), 4032, msg_h.data_ptr(), off_h.data_ptr(), None, 0, None,
                                   sig_h.data_ptr(), None, n, 0, None))

    for _ in range(warmup):
        step_device()
    cx.barrier()
    if sampler is not None and rank == 0:
        sampler.start()
    l0 = cx.cb.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step_device()
    ev1.record()
    cx.barrier()
    launches = cx.cb.launch_count() - l0
    ms_step = cx.max_over_ranks(ev0.elapsed_time(ev1) / steps)
    clocks = sampler.stop() if (sampler is not None and rank == 0) else None
    att = attempts.value / n
    assert int(st_d.sum().item()) == 0
    if dump_dir is not None and rank == 0:
        # each rank signs its own shard; rank 0's caller receives rank 0's signatures
        rows = dump_rows(n, 3309)
        dump_outputs(dump_dir, rows, {"sig": sig_d[torch.as_tensor(rows, device=sig_d.device)].cpu().numpy()})
    step_host()
    cx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host()
    e2e_ms = cx.max_over_ranks(1e3 * (time.perf_counter() - t0) / steps)
    same = bool(torch.equal(sig_h[:4096], sig_d[:4096].cpu()))
    kernels = cx.profile(step_device)
    tot = sum(v["ms_total"] for v in kernels.values())
    dom_name = max(kernels, key=lambda k_: kernels[k_]["ms_total"])
    # the dominant class runs once per round over the still-active signatures: all of its launches together
    # process the whole batch, so its per-step time is the launch duration the roofline refers to
    achieved = MLDSA["bytes_per_op"] * n / (kernels[dom_name]["ms_total"] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": cx.peak, "unit": "GB/s",
                "frac": achieved / cx.peak, "traffic": ncu_traffic(dom_name, n * att), "peak_kind": cx.peak_kind,
                "share_of_step": kernels[dom_name]["ms_total"] / tot,
                "note": "integer-ALU (Keccak + NTT) bound; achieved = 7373 algorithmic B/op x batch / time of this kernel "
                        "class summed over the rounds of one step; traffic = ncu dram bytes of the first round scaled to "
                        "all op-rounds of the step",
                "kernels_ms_per_step": {k_: round(v["ms_total"], 3) for k_, v in kernels.items()}}
    cpu = None
    if with_cpu and rank == 0 and world == 1:
        import oracle
        threads = host_threads()
        sample = 1 << 12
        sks = np.ascontiguousarray(sk_h.numpy()[:sample])
        msgs = [bytes(m) for m in msg_h.numpy()[:sample]]
        t0 = time.perf_counter()
        want, _ = oracle.mldsa65_sign_batch(sks, msgs, nthreads=threads)
        dt = time.perf_counter() - t0
        cpu = {"value": sample / dt, "unit": "sign/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} signatures of the batch, all {threads} host threads, per-op sk expansion",
               "outputs_match_gpu": bool(np.array_equal(want, sig_h.numpy()[:sample]))}
    cfg = mldsa_config(n)
    cfg["attempts_per_signature"] = att
    rec = {"metric": "ML-DSA-65 sign/sec", "value": world * n / (ms_step * 1e-3), "unit": "sign/s",
           "ms_per_step": ms_step, "dtype": "uint32", "config": cfg,
           "e2e": {"value": world * n / (e2e_ms * 1e-3), "unit": "sign/s", "ms_per_step": e2e_ms,
                   "h2d_bytes_per_step": n * (4032 + 32 + 8), "d2h_bytes_per_step": n * 3310,
                   "host_vs_device_outputs_equal": same},
           "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu}
    del sk_d, sig_d, sk_h, sig_h
    torch.cuda.empty_cache()
    return rec, clocks


# ---------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mlkem768", choices=list(WORKLOADS) + ["mldsa65"])
    ap.add_argument("--batch-log2", type=int, default=20, help="operations per GPU = 2^this")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ntt", action="store_true", help="skip the secondary NTT / Keccak measurements")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra BASELINE configs (mldsa65 at N = 1, mlkem1024 at N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (a fixed sample of its rows) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_mldsa(args) if args.workload == "mldsa65" else run_reference(args)

    cx = Ctx(args)
    sampler = ClockSampler(cx.local)
    with_cpu = not args.no_cpu_baseline
    common = {"n_gpus": cx.world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
              "vs_baseline": None, "data": "synthetic"}
    if args.workload == "mldsa65":
        log2 = args.batch_log2 if args.batch_log2 != 20 else 18
        rec, clocks = bench_mldsa(cx, log2, args.steps, args.warmup, with_cpu, sampler, args.dump_outputs)
        line = dict(rec, **common, clocks=clocks)
    else:
        rec, clocks = bench_mlkem(cx, args.workload, args.batch_log2, args.steps, args.warmup, True, with_cpu, args.steps,
                                  sampler, args.dump_outputs)
        line = dict(rec, **common, dtype="int16", clocks=clocks)
        line.pop("per_gpu", None)
        if not args.no_ntt:
            line["ntt"] = bench_ntt(cx, args.steps, args.warmup, with_cpu)
            line["keccak"] = bench_keccak(cx, args.steps, args.warmup)
        if not args.no_extras and args.workload == "mlkem768" and args.batch_log2 == 20:
            if cx.world == 1:
                line["mldsa65"], _ = bench_mldsa(cx, 18, args.steps, 3, with_cpu)
            else:
                # BASELINE configs[4]: 2^21 per GPU = 2^24 over 8 GPUs, gathered to rank 0 (26.8 GB at N = 8)
                line["mlkem1024"], _ = bench_mlkem(cx, "mlkem1024", 21, args.steps, 3, with_profile=False,
                                                   with_cpu=False, e2e_steps=args.steps)
    if cx.rank == 0:
        print(json.dumps(line))
    if cx.world > 1:
        cx.dist.destroy_process_group()
    cx.cb.shutdown()
    return 0


if __name__ == "__main__":
    sys.exit(main())
