#!/usr/bin/env python3
"""bench.py — headline benchmark of the hot path (BASELINE.json): secp256r1 prj_pt_mul/s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Default workload (N = 1) is BASELINE.json
configs[1]: 2^20 random scalars on the fixed base G of secp256r1 per GPU.  The other configs of BASELINE.json
(frp256v1_ecdsa_verify = config 3, secp384r1_fixed_base = config 4, the variable-base form, config 5's 2^24 over 8
GPUs) are measured by the same code on short runs and reported in the `extra` block of the same JSON line.

Ours arm, per step and per rank (one process per GPU; torchrun for N > 1) — the SAME timing protocol at every N:
  value  : inputs resident in HBM, eccb200_*_batch_dev on torch's current stream; per-step CUDA events with the L2
           flush between steps outside them; sum over the K steps, max over ranks.  For N > 1 the step includes the
           result gather (--gather peer-root, default): a copy-engine push of every rank's results into rank 0's
           gathered buffer over NVLink (peer-mapped memory), pipelined one step behind the kernels, the last push waited
           for inside the timed region; peer-all = every rank receives everything; fused-* = the normalisation kernel
           stores into the peers itself; nccl = one all_gather per step.
  e2e    : the host-pointer C-ABI call (eccb200_prj_pt_mul_batch / eccb200_ecdsa_verify_msgs_batch) on host buffers:
           host->device copy of the step's inputs and device->host copy of its results inside the timed region.
  roofline: the dominant kernel's own duration (CUDA events recorded by the library around that kernel on the
           launching stream) against the measured integer multiply-add peak (imad_peak micro-benchmark, run here).
  cpu_baseline: the unmodified reference (oracle/_ref/libecc_ref.so, kind "reference") on this box's host cores on a
           bounded prefix of the same inputs (rank 0, N = 1).

Reference arm (--impl reference): the reference's own CPU implementation of the path (oracle/_ref, else the oracle
port) on all host cores, each step a bounded sample of the same workload; rank 0 only.

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned to its caller as float32
.npy files (inputs are seeded, so two builds run with the same arguments can be compared output for output):
verdicts.npy (one per item) for the verification workloads; points.npy (affine x || y bytes) and status.npy for the
scalar multiplications, on a fixed seeded sample of DUMP_ITEMS items whose positions are in sample_index.npy.
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (curve, kind, metric name, unit)
    "secp256r1_fixed_base": ("SECP256R1", "fixed", "secp256r1 prj_pt_mul/sec", "prj_pt_mul/s"),
    "secp384r1_fixed_base": ("SECP384R1", "fixed", "secp384r1 prj_pt_mul/sec", "prj_pt_mul/s"),
    "frp256v1_fixed_base": ("FRP256V1", "fixed", "frp256v1 prj_pt_mul/sec", "prj_pt_mul/s"),
    "secp256r1_variable_base": ("SECP256R1", "var", "secp256r1 variable-base prj_pt_mul/sec", "prj_pt_mul/s"),
    "frp256v1_ecdsa_verify": ("FRP256V1", "verify", "frp256v1 ECDSA ec_verify/sec", "ec_verify/s"),
    "secp256r1_ecdsa_verify": ("SECP256R1", "verify", "secp256r1 ECDSA ec_verify/sec", "ec_verify/s"),
    "brainpoolp256r1_fixed_base": ("BRAINPOOLP256R1", "fixed", "brainpoolp256r1 prj_pt_mul/sec", "prj_pt_mul/s"),
    "brainpoolp256r1_ecdsa_verify": ("BRAINPOOLP256R1", "verify", "brainpoolp256r1 ECDSA ec_verify/sec", "ec_verify/s"),
    "secp256k1_fixed_base": ("SECP256K1", "fixed", "secp256k1 prj_pt_mul/sec", "prj_pt_mul/s"),
    "secp521r1_fixed_base": ("SECP521R1", "fixed", "secp521r1 prj_pt_mul/sec", "prj_pt_mul/s"),
    "secp521r1_variable_base": ("SECP521R1", "var", "secp521r1 prj_pt_mul/sec (variable base)", "prj_pt_mul/s"),
    "secp521r1_ecdsa_verify": ("SECP521R1", "verify", "secp521r1 ECDSA ec_verify/sec", "ec_verify/s"),
}
SEED = 0x6C69626563632D31
SETTLE_STEPS = 10     # untimed steps after the W warm-up steps (see Ours.measure_device)
MSG_LEN = 32          # the ECDSA workloads verify MESSAGES (ec_verify hashes them): 32 random bytes each, SHA-256
VERIFY_HASH = "SHA256"
# comb window of the fixed-base table when --comb-window is not given: the widest table that pays on a B200
# (measured sweep in DESIGN.md §4); other curves keep the library default
# round 2, one B200, 2^20 scalars: secp256r1 w = 22 / 24 / 26 -> 513 / 555 / 604 M/s (tables 3.2 / 11.8 / 40 GiB of the
# 180 GB HBM); secp384r1 keeps to 24 bits (24 GiB; 26 bits would be 90 GiB)
DEFAULT_COMB = {"SECP256R1": int(os.environ.get("BENCH_COMB_WINDOW", "26")),
                "SECP384R1": int(os.environ.get("BENCH_COMB_WINDOW_384", "24"))}
# --dump-outputs keeps the files under 64 MB: 2^16 points of secp521r1 are 132 bytes, 35 MB as float32
DUMP_ITEMS = 1 << 16


def splitmix_bytes(n_bytes: int, tag: int) -> np.ndarray:
    g = np.random.default_rng([SEED & 0xFFFFFFFF, SEED >> 32, tag])
    return g.integers(0, 256, size=n_bytes, dtype=np.uint8)


def nproc() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def host_info() -> dict:
    """What the CPU numbers were measured on (the same 'cores' figure meant 5x different rates on two boxes)."""
    info = {"affinity_cpus": nproc(), "os_cpus": os.cpu_count()}
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                info["model"] = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    try:
        info["loadavg"] = [float(x) for x in open("/proc/loadavg").read().split()[:3]]
    except (OSError, ValueError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_cpu_limit"] = open(path).read().strip()
            break
        except OSError:
            continue
    # CPUs' worth of time the container may use: "<quota> <period>" in cpu.max ("max" = unlimited).  A box that shows
    # 128 hardware threads under a 16-CPU quota runs the 128 baseline threads at the rate of 16 cores: that, not the
    # thread count, sets the reference rate (4.5 k/s under a 16-CPU quota on the pool's one-GPU boxes).
    info["effective_cpus"] = float(info["affinity_cpus"])
    try:
        parts = info.get("cgroup_cpu_limit", "").split()
        if len(parts) == 2 and parts[0] != "max" and float(parts[1]) > 0:
            info["effective_cpus"] = min(info["effective_cpus"], float(parts[0]) / float(parts[1]))
        elif len(parts) == 1 and parts[0] not in ("max", "-1") and float(parts[0]) > 0:   # cgroup v1 quota, 100 ms period
            info["effective_cpus"] = min(info["effective_cpus"], float(parts[0]) / 100000.0)
    except ValueError:
        pass
    return info


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason sampling during the timed region (NVML, ~5 ms period)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop_evt.wait(0.004)   # the timed region of the default run lasts ~20 ms

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ inputs

def make_scalars(curve: str, n: int, tag: int) -> np.ndarray:
    """Seeded scalars of SURVEY.md §8d: uniform in [1, q-1] plus ~0.1 % edge scalars (0, 1, q-1, q, q+1, 2^l-1, ...)."""
    from common import ALL_CURVES as CURVES, ORDER, edge_scalars
    _, plen, qlen = CURVES[curve]
    q = ORDER[curve]
    raw = splitmix_bytes(n * qlen, tag).reshape(n, qlen)
    raw[:, 0] &= (1 << (q.bit_length() - 8 * (qlen - 1))) - 1   # bitlen(q) need not be a multiple of 8 (P-521)
    vals_hi = raw[:, 0].astype(np.int64)
    qb = np.frombuffer(q.to_bytes(qlen, "big"), dtype=np.uint8)
    suspicious = np.nonzero(vals_hi >= int(qb[0]))[0]           # rejection on the few rows that could be >= q
    g = np.random.default_rng(7 + tag)
    for i in suspicious:
        while not (0 < int.from_bytes(raw[i].tobytes(), "big") < q):
            raw[i] = g.integers(0, 256, size=qlen, dtype=np.uint8)
            raw[i, 0] &= (1 << (q.bit_length() - 8 * (qlen - 1))) - 1
    es = edge_scalars(curve)
    slots = np.arange(0, n, 1024)[: max(1, n // 1024)]
    raw[slots] = es[np.arange(len(slots)) % es.shape[0]]
    return np.ascontiguousarray(raw)


def make_inputs(workload: str, n: int, rank: int, use_gpu: bool = True):
    """Seeded synthetic inputs for one rank (host numpy arrays).  Fixed / variable base: TWO scalar sets, used by
    alternate steps so that consecutive steps do not gather the same table entries."""
    curve, kind, _, _ = WORKLOADS[workload]
    inputs = {"scalars": make_scalars(curve, n, 100 + rank)}
    if kind in ("fixed", "var"):
        inputs["scalars_b"] = make_scalars(curve, n, 4100 + rank)
    if kind == "var":
        inputs["points"] = make_points(curve, n, rank)
    if kind == "verify":
        inputs.update(make_verify_inputs(curve, n, rank, use_gpu))
    return inputs


def make_points(curve: str, n: int, rank: int) -> np.ndarray:
    """n distinct valid affine points: produced by the engine's own fixed-base path from seeded scalars and
    spot-checked against the oracle (the reference would need minutes for 2^20 points)."""
    import libecc_b200
    from common import ALL_CURVES, ORDER, oracle_smul
    qlen = ALL_CURVES[curve][2]
    sc = splitmix_bytes(n * qlen, 300 + rank).reshape(n, qlen)
    sc[:, 0] &= ((1 << (ORDER[curve].bit_length() - 8 * (qlen - 1))) - 1) >> 1   # < q without rejection
    eng = libecc_b200.Engine(curve, device=int(os.environ.get("LOCAL_RANK", 0)), comb_window=16)
    pts, st = eng.prj_pt_mul_batch(sc)
    assert (st == 0).all()
    want, _ = oracle_smul(curve, sc[:64])
    assert (pts[:64] == want).all()
    eng.close()
    return pts


def sha256_rows(msgs: np.ndarray) -> np.ndarray:
    return np.frombuffer(b"".join(hashlib.sha256(m.tobytes()).digest() for m in msgs), dtype=np.uint8) \
        .reshape(len(msgs), 32).copy()


def make_verify_inputs(curve: str, n: int, rank: int, use_gpu: bool = True):
    """(sigs, pubkeys, msgs, digests, expected) of SURVEY.md §8d.3: a distinct random key and a distinct random 32-byte
    message per tuple, 1/16 of the tuples corrupted (bit flip in r, s, message or key; r = 0; s = q) with the expected
    verdict recorded.  Ours arm: digests, keys and signatures come from the engine's own batch entry points (device
    SHA-256, d*G, then r, s); a 2^12 sample is cross-checked with hashlib and the oracle's signer and verifier.
    Reference arm (no GPU): hashlib + the oracle's signer on a 2^12 pool, tiled."""
    from common import ALL_CURVES as CURVES, ORDER, oracle_sign, oracle_smul, oracle_verify, random_scalars
    _, plen, qlen = CURVES[curve]
    hlen = 32
    q = ORDER[curve]
    qbytes = np.frombuffer(q.to_bytes(qlen, "big"), dtype=np.uint8)

    def corrupt(sigs, pubs, msgs, count):
        expected = np.zeros(count, dtype=np.int8)
        idx = np.arange(0, count, 16)
        kind = (idx // 16) % 6
        expected[idx] = -1
        sigs[idx[kind == 0], qlen - 1] ^= 1              # bit flip in r
        sigs[idx[kind == 1], 2 * qlen - 1] ^= 1          # bit flip in s
        msgs[idx[kind == 2], 0] ^= 0x80                  # bit flip in the message
        pubs[idx[kind == 3], plen - 1] ^= 1              # key off the curve
        sigs[idx[kind == 4], :qlen] = 0                  # r = 0
        sigs[idx[kind == 5], qlen:] = qbytes             # s = q
        return expected

    if not use_gpu:
        pool = min(1 << 12, n)
        msgs = splitmix_bytes(pool * MSG_LEN, 800 + rank).reshape(pool, MSG_LEN)
        d = random_scalars(curve, pool, tag=1500 + rank)
        k = random_scalars(curve, pool, tag=2500 + rank)
        pubs, st = oracle_smul(curve, d)
        sigs, st = oracle_sign(curve, d, k, sha256_rows(msgs), hlen)
        expected = corrupt(sigs, pubs, msgs, pool)
        assert (oracle_verify(curve, sigs, pubs, sha256_rows(msgs), hlen) == expected).all()
        reps = (n + pool - 1) // pool
        tile = lambda a: np.ascontiguousarray(np.tile(a, (reps, 1))[:n])
        return {"sigs": tile(sigs), "pubkeys": tile(pubs), "msgs": tile(msgs), "expected": np.tile(expected, reps)[:n].copy(),
                "hlen": hlen}
    import libecc_b200
    d = splitmix_bytes(n * qlen, 600 + rank).reshape(n, qlen)
    k = splitmix_bytes(n * qlen, 700 + rank).reshape(n, qlen)
    safe = ((1 << (q.bit_length() - 8 * (qlen - 1))) - 1) >> 1   # 0x7F for byte-aligned orders, 0 for P-521
    d[:, 0] &= safe
    k[:, 0] &= safe
    d[:, -1] |= 1
    k[:, -1] |= 1                                   # in [1, q-1]: top bit clear, never zero
    msgs = splitmix_bytes(n * MSG_LEN, 800 + rank).reshape(n, MSG_LEN)
    off = np.arange(n + 1, dtype=np.uint64) * MSG_LEN
    eng = libecc_b200.Engine(curve, device=int(os.environ.get("LOCAL_RANK", 0)), comb_window=16)
    dg = eng.hash_batch_raw(VERIFY_HASH, msgs, off)
    pubs, st = eng.prj_pt_mul_batch(d)
    assert (st == 0).all()
    sigs, st = eng.ecdsa_sign_batch(d, k, dg, hlen)
    assert (st == 0).all()
    eng.close()
    m = min(n, 1 << 12)                              # cross-check of the hashing and of the signer on a 2^12 sample
    assert (dg[:m] == sha256_rows(msgs[:m])).all()
    want, wst = oracle_sign(curve, d[:m], k[:m], dg[:m], hlen)
    assert (wst == 0).all() and (want == sigs[:m]).all()
    expected = corrupt(sigs, pubs, msgs, n)
    changed = np.arange(0, n, 16)[(np.arange(0, n, 16) // 16) % 6 == 2]      # rows whose message was corrupted
    dg[changed] = sha256_rows(msgs[changed])
    assert (oracle_verify(curve, sigs[:m], pubs[:m], sha256_rows(msgs[:m]), hlen) == expected[:m]).all()
    return {"sigs": sigs, "pubkeys": pubs, "msgs": msgs, "digests_host": dg, "expected": expected, "hlen": hlen}


def dump_outputs(path: str, kind: str, results) -> None:
    """--dump-outputs: the last timed step's results, (verdicts,) or (points, status), as float32 .npy files."""
    os.makedirs(path, exist_ok=True)
    save = lambda name, a: np.save(os.path.join(path, name + ".npy"), np.asarray(a).astype(np.float32))
    if kind == "verify":
        save("verdicts", results[0])
        return
    out, st = results
    n = out.shape[0]
    idx = np.sort(np.random.default_rng(SEED).choice(n, size=min(n, DUMP_ITEMS), replace=False))
    np.save(os.path.join(path, "sample_index.npy"), idx.astype(np.float64))
    save("points", out[idx])
    save("status", st[idx])


# ------------------------------------------------------------------------------------------------ CPU arms

def ref_lib():
    path = os.path.join(ROOT, "oracle", "_ref", "libecc_ref.so")
    return ctypes.CDLL(path) if os.path.exists(path) else None


def cpu_run(workload: str, inputs, lo: int, cnt: int, threads: int):
    """Runs items [lo, lo+cnt) of the workload on the reference (or the oracle port) with `threads` host threads.
    Returns (seconds, kind, outputs)."""
    from common import ALL_CURVES as CURVES, oracle_lib
    curve, kind, _, _ = WORKLOADS[workload]
    _, plen, qlen = CURVES[curve]
    ref = ref_lib()
    ptr = lambda a: np.ascontiguousarray(a).ctypes.data_as(ctypes.c_void_p)
    if kind in ("fixed", "var"):
        sc = np.ascontiguousarray(inputs["scalars"][lo:lo + cnt])
        pts = np.ascontiguousarray(inputs["points"][lo:lo + cnt]) if kind == "var" else None
        out = np.zeros((cnt, 2 * plen), dtype=np.uint8)
        st = np.zeros(cnt, dtype=np.int8)
        t0 = time.perf_counter()
        if ref is not None:
            ref.ref_prj_pt_mul_batch(curve.encode(), cnt, ptr(sc), qlen, ptr(pts) if pts is not None else None,
                                     ptr(out), ptr(st), threads)
            k = "reference"
        else:
            oracle_lib().ora_prj_pt_mul_batch(curve.encode(), cnt, ptr(sc), qlen,
                                              ptr(pts) if pts is not None else None, ptr(out), ptr(st), threads)
            k = "port"
        return time.perf_counter() - t0, k, (out, st)
    sg = np.ascontiguousarray(inputs["sigs"][lo:lo + cnt])
    pk = np.ascontiguousarray(inputs["pubkeys"][lo:lo + cnt])
    ms = np.ascontiguousarray(inputs["msgs"][lo:lo + cnt])
    v = np.zeros(cnt, dtype=np.int8)
    if ref is not None:
        # the reference's own ec_verify on the MESSAGES: key import, SHA-256, verification (src/sig/sig_algs.c:655)
        off = np.arange(cnt + 1, dtype=np.uint64) * MSG_LEN
        t0 = time.perf_counter()
        ref.ref_ecdsa_verify_batch(curve.encode(), VERIFY_HASH.encode(), cnt, ptr(sg), ptr(pk), ptr(ms), ptr(off), ptr(v),
                                   threads)
        return time.perf_counter() - t0, "reference", (v,)
    t0 = time.perf_counter()
    dg = sha256_rows(ms)                  # the port takes digests: hashing timed with it
    oracle_lib().ora_ecdsa_verify_digest_batch(curve.encode(), cnt, ptr(sg), ptr(pk), ptr(dg), inputs["hlen"], ptr(v),
                                               threads)
    return time.perf_counter() - t0, "port", (v,)


def cpu_baseline(workload: str, inputs, budget_s: float = 12.0):
    threads = nproc()
    n = inputs["scalars"].shape[0]
    probe = min(n, 8 * threads)
    t, kind, _ = cpu_run(workload, inputs, 0, probe, threads)
    rate = probe / t
    cnt = int(min(n, max(probe, rate * budget_s)))
    t, kind, outs = cpu_run(workload, inputs, 0, cnt, threads)
    return {"value": cnt / t, "unit": WORKLOADS[workload][3], "cores": threads, "kind": kind,
            "sample": f"first {cnt} items of the step's batch, {t:.1f} s on {threads} threads",
            "host": host_info()}, cnt, outs


def ncu_dram_traffic(workload: str, batch_log2: int, comb_window: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed
    `ncu --set full` capture of this exact configuration (profiles/); None when no capture matches."""
    table = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        entries = json.load(open(table))
    except (OSError, ValueError):
        return None
    for e in entries:
        if e["workload"] == workload and e["batch_log2"] == batch_log2 and e["comb_window"] == comb_window:
            return e
    return None


def run_reference(args, rank: int):
    """--impl reference: the reference's own CPU path, bounded sample per step, rank 0 only."""
    if rank != 0:
        return
    curve, kind, metric, unit = WORKLOADS[args.workload]
    n = 1 << args.batch_log2
    # this arm times the reference's CPU path on the repo arm's workload: the same `config` object as that arm prints
    world = max(1, args.gpus)
    comb = args.comb_window or DEFAULT_COMB.get(curve, 0) or ENGINE_DEFAULT_COMB
    config = line_config(args.workload, args.batch_log2, world, comb, resolve_gather(kind, world, args.gather))
    if kind == "var":
        # no GPU on this arm: derive the points with the CPU oracle on the bounded sample only
        from common import oracle_smul
        inputs = {"scalars": make_scalars(curve, n, 100)}
        m = min(n, 1 << 12)
        pts, _ = oracle_smul(curve, splitmix_bytes(m * 32, 300).reshape(m, 32) & 0x7F)
        inputs["points"] = np.tile(pts, ((n + m - 1) // m, 1))[:n]
    else:
        inputs = make_inputs(args.workload, n, 0, use_gpu=False)
    threads = nproc()
    probe = min(n, 8 * threads)
    t, k, _ = cpu_run(args.workload, inputs, 0, probe, threads)
    # bounded sample: ~10 s of CPU work per step, less when many steps are asked for (whole run <= ~2-3 min)
    step_s = max(1.0, min(10.0, 120.0 / max(1, args.steps)))
    per_step = int(min(n, max(probe, (probe / t) * step_s)))
    per_step = min(n, 1 << max(per_step.bit_length() - 1, 0))   # a power of two: the sample size is stable across runs
    for _ in range(min(args.warmup, 1)):
        cpu_run(args.workload, inputs, 0, min(per_step, 4 * probe), threads)
    times = []
    for s in range(args.steps):
        lo = (s * per_step) % max(1, n - per_step + 1)
        t, k, outs = cpu_run(args.workload, inputs, lo, per_step, threads)
        times.append(t)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, kind, outs)
    val = per_step * len(times) / sum(times)
    line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * sum(times) / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic", "config": config,
            "cpu_baseline": {"value": val, "unit": unit, "cores": threads, "kind": k,
                             "sample": f"{per_step} items per step (bounded sample of the 2^{args.batch_log2} batch)",
                             "host": host_info()},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def workload_config(workload: str, batch_log2: int, world: int) -> dict:
    curve = WORKLOADS[workload][0]
    n = 1 << batch_log2
    return {"workload": f"{workload}: 2^{batch_log2} items per GPU per step, seeded synthetic "
                        f"(uniform scalars in [1,q-1] + 0.1% edge scalars)",
            "curve": curve, "batch_per_gpu": n, "global_batch": n * world}


ENGINE_DEFAULT_COMB = 22   # the library's default fixed-base window (eccb200_ctx_create with comb_window = 0)
_CE_DESC = ("every rank's normalisation kernel writes its results locally; a copy-engine transfer on a side stream "
            "(cudaMemcpyAsync to CUDA-IPC peer memory over NVLink, no SM involved) pushes them into {dst} gathered "
            "buffer while the NEXT step's kernels run, then publishes an arrival counter; the destination waits for "
            "step s-1's arrivals at the end of step s and for the last step's inside the timed region (drain); "
            "double-buffered with acknowledgements; no collective kernel")
GATHER_DESC = {"none": "none", "fused-root": "fused into the normalisation kernel (stores straight into rank 0's buffer)",
               "fused-all": "fused into the normalisation kernel (stores into every rank's buffer)",
               "peer-root": _CE_DESC.format(dst="rank 0's"),
               "peer-all": _CE_DESC.format(dst="every rank's"),
               "nccl": "one nccl all_gather per step on the compute stream, inside the step's events"}


def resolve_gather(kind: str, world: int, gather: str) -> str:
    """The result-gather mode a run uses (Ours.__init__): none on one GPU, NCCL for the one-byte verdicts."""
    return gather if (world > 1 and kind != "verify") else ("nccl" if world > 1 else "none")


def line_config(workload: str, batch_log2: int, world: int, comb_window: int, gather: str) -> dict:
    """The `config` object of the JSON line - the SAME for the repo arm and for `--impl reference`, which times the
    reference's CPU path on this arm's workload (the device-side entries describe the repo arm's run)."""
    return dict(workload_config(workload, batch_log2, world),
                l2="256 MiB buffer rewritten between timed iterations (outside the per-step events, at every N)",
                comb_window=comb_window, result_gather=GATHER_DESC[gather],
                timing="sum of per-step CUDA-event intervals on the compute stream, max over ranks",
                settle_steps=SETTLE_STEPS)


# ------------------------------------------------------------------------------------------------ ours

class Ours:
    """One workload on this rank's GPU: device-resident leg (`value`), host-pointer leg (`e2e`), parity checks."""

    def __init__(self, workload: str, batch_log2: int, comb_window: int, rank: int, world: int, local_rank: int,
                 gather: str):
        import torch
        import libecc_b200
        from common import ALL_CURVES as CURVES
        self.torch = torch
        self.workload, self.batch_log2 = workload, batch_log2
        self.curve, self.kind, self.metric, self.unit = WORKLOADS[workload]
        self.n = 1 << batch_log2
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.gather = resolve_gather(self.kind, world, gather)
        if world == 1 and os.environ.get("BENCH_FORCE_GATHER") and self.kind != "verify" and gather.startswith("peer"):
            self.gather = gather     # diagnostic: the gather path with this GPU as its own (only) destination
        _, self.plen, self.qlen = CURVES[self.curve]
        self.dev = torch.device("cuda", local_rank)
        self.inputs = make_inputs(workload, self.n, rank)
        if not comb_window:
            comb_window = DEFAULT_COMB.get(self.curve, 0)
        self.eng = libecc_b200.Engine(self.curve, device=local_rank, comb_window=comb_window)
        n, plen = self.n, self.plen
        skip = ("expected", "digests_host")
        self.d = {k: torch.from_numpy(v).to(self.dev) for k, v in self.inputs.items()
                  if isinstance(v, np.ndarray) and k not in skip}
        if self.kind == "verify":
            self.d["offsets"] = (torch.arange(n + 1, dtype=torch.int64, device=self.dev) * MSG_LEN)
            self.d["digests"] = torch.empty(n * 32, dtype=torch.uint8, device=self.dev)
            self.d_out = torch.empty(n, dtype=torch.int8, device=self.dev)
            self.d_status = None
            self.out_item = 1
            self.in_item = 2 * self.qlen + 2 * plen + MSG_LEN + 8
        else:
            self.d_out = torch.empty(n * 2 * plen, dtype=torch.uint8, device=self.dev)
            self.d_status = torch.empty(n, dtype=torch.int8, device=self.dev)
            self.out_item = 2 * plen + 1
            self.in_item = self.qlen + (2 * plen if self.kind == "var" else 0)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
        self.pg = None
        self.step_no = 0
        self.last_buf = 0
        if self.gather.startswith(("peer", "fused")):
            from libecc_b200.sharding import PeerGather
            self.pg = PeerGather(self.eng, rank, world, n, mode="root" if self.gather.endswith("root") else "all",
                                 transport="ce" if self.gather.startswith("peer") else "fused")
        elif self.gather == "nccl":
            out_rec = 1 if self.kind == "verify" else 2 * plen
            self.res_bytes = n * out_rec + (0 if self.kind == "verify" else n)
            self.res = torch.empty(self.res_bytes, dtype=torch.uint8, device=self.dev)
            self.gathered = torch.empty(world * self.res_bytes, dtype=torch.uint8, device=self.dev)

    # one step of the device-resident leg on torch's current stream
    def step_dev(self):
        torch, eng, d, n = self.torch, self.eng, self.d, self.n
        stream = torch.cuda.current_stream().cuda_stream
        sc = d["scalars_b"] if (self.step_no & 1 and "scalars_b" in d) else d.get("scalars")
        self.step_no += 1
        if self.kind == "verify":
            out = self.res[:n].view(torch.int8) if self.gather == "nccl" else self.d_out
            eng.ecdsa_verify_msgs_batch_dev(VERIFY_HASH, d["sigs"].view(-1), d["pubkeys"].view(-1), d["msgs"].view(-1),
                                            d["offsets"], d["digests"], out, stream)
        elif self.pg is not None:
            pts = d["points"].data_ptr() if self.kind == "var" else None
            if self.pg.transport == "ce":
                self.last_buf = self.pg.step_ce(sc.data_ptr(), pts, self.dev)
            else:
                self.last_buf = self.pg.step(sc.data_ptr(), pts, self.d_out.data_ptr(), self.d_status.data_ptr(), stream)
        else:
            if self.gather == "nccl":
                out, st = self.res[: n * 2 * self.plen], self.res[n * 2 * self.plen:].view(torch.int8)
            else:
                out, st = self.d_out, self.d_status
            eng.prj_pt_mul_batch_dev(sc.view(-1), d["points"].view(-1) if self.kind == "var" else None, out, st, stream)
        if self.gather == "nccl":     # the path's exchange step as a collective: same stream, inside the step's events
            import torch.distributed as dist
            dist.all_gather_into_tensor(self.gathered, self.res)

    def p2p_probe(self):
        """Diagnostic (BENCH_P2P_PROBE=1, N > 1, copy-engine gather): every non-root rank in turn, alone, pushes its slot
        to rank 0 five times; returns the GB/s per rank (rank 0: 0)."""
        import torch.distributed as dist
        torch = self.torch
        pg, n = self.pg, self.n
        used = n * 2 * self.plen + n
        rate = 0.0
        from libecc_b200.sharding import slot_offset
        for r in range(1, self.world):
            dist.barrier()
            torch.cuda.synchronize()
            if self.rank == r and pg is not None and 0 in pg.peer:
                src = torch.empty(used, dtype=torch.uint8, device=self.dev)
                st = torch.cuda.Stream(device=self.dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                dst = pg.peer[0] + slot_offset(pg.layout, 0, r)
                scratch_flag = pg.base + 3072          # a word of the own flag page nobody reads
                for it in range(6):
                    if it == 1:
                        e0.record(st)
                    self.eng.push_results([dst], src.data_ptr(), used, [scratch_flag], 1, None, 0, 0, st.cuda_stream)
                e1.record(st)
                st.synchronize()
                rate = 5 * used / (e0.elapsed_time(e1) / 1000.0) / 1e9
        dist.barrier()
        t = torch.tensor([rate], dtype=torch.float64, device=self.dev)
        out = [torch.zeros_like(t) for _ in range(self.world)]
        dist.all_gather(out, t)
        return [round(float(x.item()), 1) for x in out]

    def sync_all(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()

    def measure_device(self, steps: int, warmup: int) -> dict:
        torch, eng = self.torch, self.eng
        eng.profile_enable(True)
        # W warm-up steps as asked, plus SETTLE_STEPS more untimed ones: the timed region of the default run is ~30 ms, short
        # enough for a clock ramp or a lazily established peer mapping to show in it (reported as config.settle_steps)
        for _ in range(warmup + SETTLE_STEPS):
            self.step_dev()
            self.flush.zero_()
        self.sync_all()
        eng.profile_read()                      # discard the warm-up calls' timings
        launches0 = eng.kernel_launches
        sampler = ClockSampler(self.local_rank)
        sampler.start()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        kernel_ms = []
        for s in range(steps):
            self.flush.zero_()                  # L2 flush between timed iterations, outside the step's events
            evs[s][0].record()
            self.step_dev()
            evs[s][1].record()
            if (s & 7) == 7:                        # reading waits for the kernels: let the host run 8 steps ahead
                kernel_ms.append(eng.profile_read())
        drain = None
        if self.pg is not None and self.pg.transport == "ce":
            # the pushes are pipelined one step behind the kernels: the last one is waited for inside the timed region
            drain = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            drain[0].record()
            self.pg.drain(self.dev)
            drain[1].record()
        rest = eng.profile_read()
        if rest:
            kernel_ms.append(rest)
        self.sync_all()
        clocks = sampler.stop()
        step_ms = [a.elapsed_time(b) for a, b in evs]          # per-step events: the flush is outside them, at every N
        if drain is not None:
            step_ms[-1] += drain[0].elapsed_time(drain[1])
        total = torch.tensor([sum(step_ms)], dtype=torch.float64, device=self.dev)
        k2_ms = sum(k[1] for k in kernel_ms if len(k) > 1) / steps
        k1 = torch.tensor([sum(k[0] for k in kernel_ms if k) / steps, k2_ms, sum(step_ms) / steps], dtype=torch.float64,
                          device=self.dev)
        per_rank = None
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(total, op=dist.ReduceOp.MAX)
            k1_list = [torch.zeros_like(k1) for _ in range(self.world)]
            dist.all_gather(k1_list, k1)
            per_rank = {"kernel_ms": [float(x[0].item()) for x in k1_list],
                        "normalisation_ms": [float(x[1].item()) for x in k1_list],
                        "step_ms": [float(x[2].item()) for x in k1_list]}
        total_ms = float(total.item())
        return {"total_ms": total_ms, "ms_per_step": total_ms / steps, "step_ms_this_rank": step_ms,
                "value": self.n * self.world * steps / (total_ms / 1000.0), "kernel_ms": float(k1[0].item()),
                "normalisation_ms": k2_ms, "kernel_ms_per_rank": per_rank, "launches": int(eng.kernel_launches - launches0),
                "clocks": clocks, "steps": steps}

    def local_results(self):
        """Host copies of this rank's results of the LAST step (out, status) / (verdict,)."""
        torch, n = self.torch, self.n
        if self.gather == "nccl":
            if self.kind == "verify":
                return (self.res[:n].view(torch.int8).cpu().numpy(),)
            return (self.res[: n * 2 * self.plen].cpu().numpy().reshape(n, 2 * self.plen),
                    self.res[n * 2 * self.plen:].view(torch.int8).cpu().numpy())
        if self.kind == "verify":
            return (self.d_out.cpu().numpy(),)
        if self.pg is not None and self.pg.transport == "ce":     # the kernels wrote into the gather's own buffers
            raw = self.eng.copy_to_host(self.pg.last_src, n * 2 * self.plen + n)
            return raw[: n * 2 * self.plen].reshape(n, 2 * self.plen), raw[n * 2 * self.plen:].view(np.int8)
        return self.d_out.cpu().numpy().reshape(n, 2 * self.plen), self.d_status.cpu().numpy()

    def ensure_last_step_used_set_a(self):
        """The CPU baseline runs on scalar set A: make the last (untimed, if needed) step use it too."""
        if self.kind != "verify" and self.last_scalars() is not self.inputs["scalars"]:
            self.step_dev()
            self.torch.cuda.synchronize()

    def close_gather(self):
        if self.pg is not None:
            self.pg.close()
            self.pg = None

    def last_scalars(self):
        return self.inputs["scalars_b"] if ((self.step_no - 1) & 1 and "scalars_b" in self.inputs) \
            else self.inputs["scalars"]

    def parity(self) -> bool:
        """Oracle spot-check of what was just timed (first 256 items of this rank); whole-batch expectation for the
        verification workloads."""
        from common import oracle_smul, oracle_verify
        res = self.local_results()
        if self.kind == "verify":
            i = self.inputs
            want = oracle_verify(self.curve, i["sigs"][:256], i["pubkeys"][:256], sha256_rows(i["msgs"][:256]), i["hlen"])
            return bool((res[0][:256] == want).all() and (res[0] == i["expected"]).all())
        sc = self.last_scalars()
        want, wst = oracle_smul(self.curve, sc[:256], self.inputs["points"][:256] if self.kind == "var" else None)
        return bool((res[0][:256] == want).all() and (res[1][:256] == wst).all())

    def gather_checks(self) -> dict:
        """N > 1, rank 0: the gathered buffer must hold the other ranks' real results — checked against the oracle on
        inputs regenerated from the LAST rank's seed, and (peer gather) byte for byte against a NCCL all_gather of every
        rank's local results."""
        import torch.distributed as dist
        from common import oracle_smul
        torch, n, world = self.torch, self.n, self.world
        out = {}
        if self.kind != "fixed":
            return out
        slot = n * 2 * self.plen + n
        if self.pg is not None and self.pg.transport == "ce":
            mine = torch.from_numpy(self.eng.copy_to_host(self.pg.last_src, slot)).to(self.dev)
        else:
            mine = torch.cat([self.d_out if self.gather != "nccl" else self.res[: n * 2 * self.plen],
                              (self.d_status if self.gather != "nccl" else self.res[n * 2 * self.plen:].view(torch.int8))
                              .view(torch.uint8)])
        via_nccl = torch.empty(world * slot, dtype=torch.uint8, device=self.dev)
        dist.all_gather_into_tensor(via_nccl, mine)            # outside every timed region
        torch.cuda.synchronize()
        if self.rank != 0:
            return out
        if self.pg is not None:
            got = np.concatenate([self.eng.copy_to_host(self.pg.buffer_ptr(self.last_buf, r), slot) for r in range(world)])
            out["gather_matches_nccl"] = bool((got == via_nccl.cpu().numpy()).all())
        else:
            got = self.gathered.cpu().numpy()
        other = world - 1
        tag = (4100 if ((self.step_no - 1) & 1) else 100) + other
        osc = make_scalars(self.curve, n, tag)[:128]
        want_o, _ = oracle_smul(self.curve, osc)
        got_o = got.reshape(world, -1)[other][: 128 * 2 * self.plen].reshape(128, 2 * self.plen)
        out["gather_parity_other_rank"] = bool((got_o == want_o).all())
        return out

    def measure_e2e(self, steps: int, n_items: int = None) -> dict:
        """The host-pointer C-ABI call on page-locked host buffers: H2D + kernels + D2H inside the timed region."""
        import libecc_b200
        torch, eng, inputs = self.torch, self.eng, self.inputs
        n = n_items or self.n
        restore = None
        if self.world == 1:
            # the page-locked buffers and the calling thread belong on the GPU's NUMA node (N > 1: the whole rank is bound)
            restore = os.sched_getaffinity(0)
            libecc_b200.load_library().eccb200_bind_thread_near_device(self.local_rank)
        reps = (n + self.n - 1) // self.n
        wc = os.environ.get("BENCH_WC_INPUTS", "0") == "1"

        def pinned_from(a):
            full = np.tile(a, (reps, 1))[:n] if reps > 1 else a
            h = libecc_b200.pinned_empty(full.shape, full.dtype, write_combined=wc)
            h[...] = full
            return h
        if self.kind == "verify":
            hp = {k: pinned_from(inputs[k]) for k in ("sigs", "pubkeys", "msgs")}
            off = libecc_b200.pinned_empty(n + 1, np.uint64)
            off[...] = np.arange(n + 1, dtype=np.uint64) * MSG_LEN
            h_verdict = libecc_b200.pinned_empty(n, np.int8)
            call = lambda: eng.ecdsa_verify_msgs_batch_raw(VERIFY_HASH, hp["sigs"], hp["pubkeys"], hp["msgs"], off,
                                                           verdict=h_verdict)
        else:
            hp = {"scalars": pinned_from(inputs["scalars"])}
            if self.kind == "var":
                hp["points"] = pinned_from(inputs["points"])
            h_out = libecc_b200.pinned_empty((n, 2 * self.plen), np.uint8)
            h_status = libecc_b200.pinned_empty(n, np.int8)
            call = lambda: eng.prj_pt_mul_batch(hp["scalars"], hp.get("points"), out=h_out, status=h_status)
        call()
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = call()
        e1.record()
        self.sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        val = n * self.world * steps / (float(ms.item()) / 1000.0)
        # the host-pointer results must equal the device leg's (which the oracle checks) on the first self.n items
        if self.kind == "verify":
            same = bool((np.asarray(res)[: self.n] == inputs["expected"]).all())
        else:
            from common import oracle_smul
            want, wst = oracle_smul(self.curve, inputs["scalars"][:256], inputs["points"][:256] if self.kind == "var" else None)
            same = bool((res[0][:256] == want).all() and (res[1][:256] == wst).all())
            if reps > 1:                                  # tiled inputs: every tile must repeat the first one
                same = same and bool((res[0][self.n: 2 * self.n] == res[0][: self.n]).all())
        if restore is not None:
            os.sched_setaffinity(0, restore)
        return {"value": val, "unit": self.unit, "h2d_bytes_per_step": n * self.in_item,
                "d2h_bytes_per_step": n * self.out_item, "steps": steps, "items_per_gpu": n,
                "host_buffers": "page-locked (eccb200_host_alloc)", "parity": same}

    def roofline(self, kernel_ms: float, step_ms: float) -> dict:
        from roofline import imad_peak_measured, work_per_item
        n = self.n
        peak = imad_peak_measured(self.local_rank)
        work = work_per_item(self.workload, self.eng.comb_window)
        traffic = ncu_dram_traffic(self.workload, self.batch_log2, self.eng.comb_window)
        hbm = None
        try:   # driver-written measured copy bandwidth of this pool's B200s
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
            if traffic:
                gbs = traffic["bytes_per_launch"] / (kernel_ms / 1000.0) / 1e9
                hbm = {"dram_GBps": gbs, "measured_peak_GBps": hbm_peak, "frac": gbs / hbm_peak,
                       "note": "DRAM bytes of the ncu capture over the kernel's live duration: far from the HBM roof, the "
                               "kernel is bound by the integer multiply-add pipe"}
        except (OSError, ValueError, KeyError):
            pass
        achieved = n * work["imad32_per_item"] / (kernel_ms / 1000.0) / 1e12
        executed = n * work["imad_executed_per_item"] / (kernel_ms / 1000.0) / 1e12
        return {"bound": "int-mad", "kernel": work["kernel"], "achieved": achieved, "peak": peak["timad32_per_s"],
                "unit": "T IMAD32/s", "frac": achieved / peak["timad32_per_s"],
                "frac_executed_imad_wide": executed / peak["timad32_per_s"],
                "frac_note": "frac charges the generic CIOS cost (SURVEY.md 8d: 4(2n^2+n) IMAD32 per product) to every "
                             "product and so can exceed 1; frac_executed_imad_wide counts the IMAD.WIDE instructions "
                             "the kernel really issues and is the figure to compare with ncu's fmaheavy pipe utilisation",
                "traffic": traffic, "hbm": hbm,
                "kernel_ms": kernel_ms, "kernel_share_of_step": kernel_ms / step_ms,
                "normalisation_kernel_ms": getattr(self, "_k4_ms", None),
                "M_impl": work["M_impl"], "imad32_per_field_mul": work["imad32_per_mul"],
                "ref_normalised_frac": n * work["imad32_ref_per_item"] / (kernel_ms / 1000.0) / 1e12 / peak["timad32_per_s"],
                "peak_source": peak["how"],
                "hbm_algorithmic_GBps": n * (self.in_item + self.out_item) / (kernel_ms / 1000.0) / 1e9}

    def close(self):
        if self.pg is not None:
            self.pg.close()
            self.pg = None
        self.eng.close()


def run_extra(name: str, batch_log2: int, steps: int, warmup: int, local_rank: int, with_cpu: bool) -> dict:
    """Short measurement of another BASELINE.json config with the same code as the headline (N = 1)."""
    t0 = time.perf_counter()
    o = Ours(name, batch_log2, 0, 0, 1, local_rank, "none")
    m = o.measure_device(steps, warmup)
    parity = o.parity()
    rl = o.roofline(m["kernel_ms"], m["ms_per_step"])
    e2e = o.measure_e2e(max(2, min(steps, 3)))
    res = {"metric": o.metric, "unit": o.unit, "value": m["value"], "ms_per_step": m["ms_per_step"], "steps": steps,
           "warmup": warmup, "batch": 1 << batch_log2, "comb_window": o.eng.comb_window, "kernel": rl["kernel"],
           "kernel_ms": m["kernel_ms"], "normalisation_ms": m["normalisation_ms"], "roofline_frac": rl["frac"], "frac_executed_imad_wide": rl["frac_executed_imad_wide"],
           "M_impl": rl["M_impl"], "parity_spot_check": parity, "e2e": {k: e2e[k] for k in
                                                                       ("value", "h2d_bytes_per_step", "d2h_bytes_per_step",
                                                                        "steps", "parity")},
           "clocks": m["clocks"]}
    if with_cpu:
        cb, cnt, outs = cpu_baseline(name, o.inputs, budget_s=4.0)
        res["cpu_baseline"] = {k: cb[k] for k in ("value", "cores", "kind", "sample")}
        o.ensure_last_step_used_set_a()
        got = o.local_results()
        if o.kind == "verify":
            res["parity_on_cpu_prefix"] = bool((got[0][:cnt] == outs[0]).all())
        else:
            res["parity_on_cpu_prefix"] = bool((got[0][:cnt] == outs[0]).all() and (got[1][:cnt] == outs[1]).all())
    o.close()
    res["wall_s"] = round(time.perf_counter() - t0, 1)
    return res


def run_sign_and_ecdh(local_rank: int, batch_log2: int = 20) -> dict:
    """End-to-end rates of the two §8f.1 / f.2 batch entry points (host pointers, page-locked buffers), each checked
    against the oracle on a prefix: ECDSA signing with caller-supplied nonces and ECC-CDH derivation (secp256r1)."""
    import libecc_b200
    from common import ALL_CURVES as CURVES, ORDER, oracle_sign, oracle_smul
    curve = "SECP256R1"
    _, plen, qlen = CURVES[curve]
    n = 1 << batch_log2
    q = ORDER[curve]
    pin = lambda a: (lambda h: (h.__setitem__(Ellipsis, a), h)[1])(libecc_b200.pinned_empty(a.shape, a.dtype))
    d = splitmix_bytes(n * qlen, 9600).reshape(n, qlen); d[:, 0] &= 0x7F; d[:, -1] |= 1
    k = splitmix_bytes(n * qlen, 9700).reshape(n, qlen); k[:, 0] &= 0x7F; k[:, -1] |= 1
    dg = splitmix_bytes(n * 32, 9800).reshape(n, 32)
    eng = libecc_b200.Engine(curve, device=local_rank, comb_window=DEFAULT_COMB.get(curve, 0))
    out = {}
    hd, hk, hdg = pin(d), pin(k), pin(dg)
    h_sig, h_st = libecc_b200.pinned_empty((n, 2 * qlen), np.uint8), libecc_b200.pinned_empty(n, np.int8)
    eng.ecdsa_sign_batch(hd, hk, hdg, 32, out=h_sig, status=h_st)
    t0 = time.perf_counter()
    for _ in range(3):
        sigs, st = eng.ecdsa_sign_batch(hd, hk, hdg, 32, out=h_sig, status=h_st)
    dt = (time.perf_counter() - t0) / 3
    want, wst = oracle_sign(curve, d[:256], k[:256], dg[:256], 32)
    out["secp256r1_ecdsa_sign"] = {"e2e_value": n / dt, "unit": "ec_sign/s (nonces supplied, digests)", "items": n,
                                   "parity_spot_check": bool((sigs[:256] == want).all() and (st[:256] == wst).all() and (st == 0).all())}
    pubs, _ = eng.prj_pt_mul_batch(k)                       # peers' public keys k_i * G
    hp = pin(pubs)
    h_sh = libecc_b200.pinned_empty((n, plen), np.uint8)
    eng.ecccdh_derive_batch(hd, hp, out=h_sh, status=h_st)
    t0 = time.perf_counter()
    for _ in range(2):
        shared, st = eng.ecccdh_derive_batch(hd, hp, out=h_sh, status=h_st)
    dt = (time.perf_counter() - t0) / 2
    want, wst = oracle_smul(curve, d[:128], pubs[:128])
    out["secp256r1_ecccdh_derive"] = {"e2e_value": n / dt, "unit": "shared secrets/s", "items": n,
                                      "parity_spot_check": bool((shared[:128] == want[:, :plen]).all() and (st == 0).all())}
    eng.close()
    return out


def run_schnorr_msm(local_rank: int, scheme: str = "ecfsdsa", batch_log2: int = 20, with_cpu: bool = True) -> dict:
    """§8f.4: Schnorr-type batch verification in the reference's verify_batch form (one random linear combination for
    the whole batch, src/sig/ecfsdsa.c:814-1055, src/sig/bip0340.c:1040-1290) as a multi-scalar multiplication on the
    device (K6), next to the per-item verification kernel on the same batch.  2^14 distinct signatures made here (k*G and
    d*G by the engine, the rest is hashlib and integers), tiled to the batch size.  ECFSDSA on FRP256V1, BIP0340 on
    SECP256K1; SHA-256."""
    import hashlib
    import torch
    import libecc_b200
    from common import ALL_CURVES as CURVES, ORDER
    bip = scheme == "bip0340"
    curve = "SECP256K1" if bip else "FRP256V1"
    _, plen, qlen = CURVES[curve]
    q = ORDER[curve]
    n, m = 1 << batch_log2, 1 << 14
    eng = libecc_b200.Engine(curve, device=local_rank, comb_window=16)
    d = splitmix_bytes(m * qlen, 9900).reshape(m, qlen); d[:, 0] &= 0x7F; d[:, -1] |= 1
    k = splitmix_bytes(m * qlen, 9901).reshape(m, qlen); k[:, 0] &= 0x7F; k[:, -1] |= 1
    msgs = splitmix_bytes(m * 32, 9902).reshape(m, 32)
    pubs, st1 = eng.prj_pt_mul_batch(d)
    W, st2 = eng.prj_pt_mul_batch(k)
    assert (st1 == 0).all() and (st2 == 0).all()
    siglen = (plen if bip else 2 * plen) + qlen
    sigs = np.zeros((m, siglen), np.uint8)
    dg = np.zeros((m, 32), np.uint8)
    sigs[:, :siglen - qlen] = W[:, :siglen - qlen]
    tag = hashlib.sha256(b"BIP0340/challenge").digest()
    for i in range(m):
        di, ki = int.from_bytes(d[i].tobytes(), "big"), int.from_bytes(k[i].tobytes(), "big")
        if bip:
            # sig/bip0340.c:239-330: the secret and the nonce are negated when their points have an odd y
            if pubs[i, -1] & 1: di = q - di
            if W[i, -1] & 1: ki = q - ki
            h = hashlib.sha256(tag + tag + W[i, :plen].tobytes() + pubs[i, :plen].tobytes() + msgs[i].tobytes()).digest()
        else:
            h = hashlib.sha256(W[i].tobytes() + msgs[i].tobytes()).digest()
        dg[i] = np.frombuffer(h, np.uint8)
        sigs[i, siglen - qlen:] = np.frombuffer(((ki + int.from_bytes(h, "big") * di) % q).to_bytes(qlen, "big"), np.uint8)
    reps = n // m
    S, P, D = np.tile(sigs, (reps, 1)), np.tile(pubs, (reps, 1)), np.tile(dg, (reps, 1))
    dev = torch.device("cuda", local_rank)
    dS, dP, dD = (torch.from_numpy(a).to(dev) for a in (S, P, D))
    dV = torch.empty(n, dtype=torch.int8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = eng.lib
    msm_dev = lib.eccb200_bip0340_verify_msm_batch_dev if bip else lib.eccb200_ecfsdsa_verify_msm_batch_dev
    item_dev = lib.eccb200_bip0340_verify_batch_dev if bip else lib.eccb200_ecfsdsa_verify_batch_dev
    msm_host = eng.bip0340_verify_msm_batch if bip else eng.ecfsdsa_verify_msm_batch

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        ms = []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.mean(ms))

    verdicts = []

    def msm():
        ok = ctypes.c_int(0)
        assert msm_dev(eng._h, n, dS.data_ptr(), dP.data_ptr(), dD.data_ptr(), 32, None, ctypes.byref(ok), stream) == 0
        verdicts.append(ok.value == 1)
    l0 = eng.kernel_launches
    ms_msm = timed(msm, 5, 2)
    launches = int(eng.kernel_launches - l0) // 7  # 5 timed + 2 warm-up calls

    def per_item():
        assert item_dev(eng._h, n, dS.data_ptr(), dP.data_ptr(), dD.data_ptr(), 32, dV.data_ptr(), stream) == 0
    ms_item = timed(per_item, 3, 1)
    item_ok = bool((dV == 0).all().item())
    # end to end through the host-pointer call (page-locked inputs), the verdict is the only output
    pin = lambda a: (lambda h: (h.__setitem__(Ellipsis, a), h)[1])(libecc_b200.pinned_empty(a.shape, a.dtype))
    hS, hP, hD = pin(S), pin(P), pin(D)
    msm_host(hS, hP, hD, 32)
    t0 = time.perf_counter()
    e2e_ok = [msm_host(hS, hP, hD, 32) for _ in range(3)]
    e2e_dt = (time.perf_counter() - t0) / 3
    # one flipped bit anywhere sinks the batch
    j = 777777 % n
    hS[j, -1] ^= 1
    forged = msm_host(hS, hP, hD, 32)
    hS[j, -1] ^= 1
    name = "BIP0340" if bip else "ECFSDSA"
    res = {"metric": f"{curve.lower()} {name} verify_batch (one multi-scalar multiplication) signatures/sec",
           "unit": "ec_verify/s", "value": n / (ms_msm * 1e-3), "ms_per_step": ms_msm, "batch": n, "steps": 5, "warmup": 2,
           "kernels_per_call": launches,
           "per_item_kernel_same_batch": {"value": n / (ms_item * 1e-3), "ms_per_step": ms_item, "all_valid": item_ok},
           "speedup_vs_per_item_kernel": ms_item / ms_msm,
           "e2e": {"value": n / e2e_dt, "h2d_bytes_per_step": int(S.nbytes + P.nbytes + D.nbytes), "d2h_bytes_per_step": 8},
           "accepts_valid_batch": bool(all(verdicts) and all(e2e_ok)), "rejects_one_flipped_bit": forged is False,
           "distinct_signatures": m}
    if with_cpu:
        from common import oracle_lib, _buf
        v = np.zeros(256, np.int8)
        fn = oracle_lib().ora_bip0340_verify_digest_batch if bip else oracle_lib().ora_ecfsdsa_verify_digest_batch
        assert fn(curve.encode(), 256, _buf(np.ascontiguousarray(sigs[:256])), _buf(np.ascontiguousarray(pubs[:256])),
                  _buf(np.ascontiguousarray(dg[:256])), 32, _buf(v), 8) == 0
        res["parity_on_cpu_prefix"] = bool((v == 0).all())
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="secp256r1_fixed_base", choices=sorted(WORKLOADS))
    ap.add_argument("--batch-log2", type=int, default=20, help="items per GPU per step (2^k)")
    ap.add_argument("--comb-window", type=int, default=0)
    ap.add_argument("--gather", default="peer-root", choices=["peer-root", "peer-all", "fused-root", "fused-all", "nccl"],
                    help="N > 1: how the per-step results are gathered (peer-*: copy-engine pushes into peer memory, "
                         "pipelined one step behind the kernels; fused-*: stores of the normalisation kernel itself)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE.json configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    numa_cpus = None
    full_affinity = os.sched_getaffinity(0)
    if world > 1:
        # one process per GPU on a two-socket box: keep this rank's host threads and pinned buffers on its GPU's node
        import libecc_b200
        numa_cpus = libecc_b200.load_library().eccb200_bind_thread_near_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    default_workload = args.workload == "secp256r1_fixed_base" and args.batch_log2 == 20
    o = Ours(args.workload, args.batch_log2, args.comb_window, rank, world, local_rank, args.gather)
    n = o.n
    p2p = o.p2p_probe() if (world > 1 and o.pg is not None and os.environ.get("BENCH_P2P_PROBE")) else None
    m = o.measure_device(args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, o.kind, o.local_results())
    parity = o.parity()
    gchk = o.gather_checks() if world > 1 else {}
    e2e_steps = max(3, min(args.steps, 10))
    e2e = o.measure_e2e(e2e_steps)

    extra = {}
    if world > 1 and default_workload and not args.no_extra and o.kind == "fixed":
        # config 5 as written (2^24 scalars over 8 GPUs = 2^21 per GPU) with the same gather, same protocol
        per_gpu_log2 = 24 - max(0, (world - 1).bit_length())
        if 20 < per_gpu_log2 <= 22:
            o5 = Ours(args.workload, per_gpu_log2, o.eng.comb_window, rank, world, local_rank, args.gather)
            m5 = o5.measure_device(5, 2)
            ok5 = o5.parity()
            g5 = o5.gather_checks()
            o5.close_gather()
            o5.close()
            extra["config5_2^24_total"] = dict({"value": m5["value"], "ms_per_step": m5["ms_per_step"], "steps": 5,
                                                "batch_per_gpu": 1 << per_gpu_log2, "global_batch": world << per_gpu_log2,
                                                "per_rank": m5["kernel_ms_per_rank"], "parity_spot_check": ok5}, **g5)

    if world > 1:
        o.close_gather()            # collective: every rank unmaps its peers' regions before anybody frees its own
    if rank != 0:
        o.close()
        if world > 1:
            dist.barrier()          # rank 0 may still be running its single-process multi-device leg
            dist.destroy_process_group()
        return

    o._k4_ms = m["normalisation_ms"]
    roofline = o.roofline(m["kernel_ms"], m["ms_per_step"])
    line = {"metric": o.metric, "value": m["value"], "unit": o.unit, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": line_config(args.workload, args.batch_log2, world, o.eng.comb_window, o.gather),
            "clocks": m["clocks"], "gpu_launches": m["launches"], "host_cpus_bound_near_gpu": numa_cpus,
            "e2e": dict(e2e, same_results_as_device_leg=e2e["parity"]),
            "roofline": roofline, "parity_spot_check": parity}
    line.update(gchk)
    if p2p is not None:
        line["p2p_push_GBps_per_rank_alone"] = p2p
    if m["kernel_ms_per_rank"]:
        line["per_rank"] = m["kernel_ms_per_rank"]
    if world == 1 and not args.no_cpu_baseline:
        cb, cnt, outs = cpu_baseline(args.workload, o.inputs)
        line["cpu_baseline"] = cb
        got = o.local_results()
        # the timed GPU results must equal the reference on the CPU-timed prefix (same scalar set as the last step)
        if o.kind == "verify":
            line["parity_on_cpu_prefix"] = bool((got[0][:cnt] == outs[0]).all())
        else:
            o.ensure_last_step_used_set_a()
            got = o.local_results()
            line["parity_on_cpu_prefix"] = bool((got[0][:cnt] == outs[0]).all() and (got[1][:cnt] == outs[1]).all())

    if default_workload and not args.no_extra:
        if world == 1:
            # end-to-end at larger batches (fill / drain amortised): same call, inputs tiled
            for lg in (22, 24):
                try:
                    r = o.measure_e2e(3, n_items=1 << lg)
                    extra[f"e2e_2^{lg}"] = {k: r[k] for k in ("value", "items_per_gpu", "steps", "parity")}
                except Exception as exc:       # noqa: BLE001 — an extra must not take the headline down
                    extra[f"e2e_2^{lg}"] = {"error": str(exc)[:200]}
            o.close()
            for name, lg, st, wu in (("frp256v1_ecdsa_verify", 20, 3, 1), ("secp384r1_fixed_base", 20, 5, 2),
                                     ("secp256r1_variable_base", 20, 3, 1)):
                try:
                    extra[name] = run_extra(name, lg, st, wu, local_rank, with_cpu=not args.no_cpu_baseline)
                except Exception as exc:       # noqa: BLE001
                    extra[name] = {"error": str(exc)[:300]}
            try:
                extra.update(run_sign_and_ecdh(local_rank))
            except Exception as exc:           # noqa: BLE001
                extra["sign_and_ecdh"] = {"error": str(exc)[:300]}
            for key, sch in (("frp256v1_ecfsdsa_verify_batch_msm", "ecfsdsa"), ("secp256k1_bip0340_verify_batch_msm", "bip0340")):
                try:
                    extra[key] = run_schnorr_msm(local_rank, sch, with_cpu=not args.no_cpu_baseline)
                except Exception as exc:       # noqa: BLE001
                    extra[key] = {"error": str(exc)[:300]}
        else:
            o.close()
            # the in-process multi-device C ABI (eccb200_multi_*): ONE host call shards 2^24 scalars over all GPUs of
            # the box, each GPU DMAs its shard's results straight into the caller's pinned output
            try:
                os.sched_setaffinity(0, full_affinity)     # the library binds its per-device worker threads itself
                extra["multi_device_c_abi"] = run_multi_abi(args.workload, world, 24)
            except Exception as exc:           # noqa: BLE001
                extra["multi_device_c_abi"] = {"error": str(exc)[:300]}
    else:
        o.close()
    if extra:
        line["extra"] = extra
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_multi_abi(workload: str, n_dev: int, total_log2: int) -> dict:
    import libecc_b200
    from common import ALL_CURVES as CURVES, oracle_smul
    curve, kind, metric, unit = WORKLOADS[workload]
    _, plen, qlen = CURVES[curve]
    n = 1 << total_log2
    base = make_scalars(curve, 1 << 20, 9100)
    reps = n >> 20
    h_sc = libecc_b200.pinned_empty((n, qlen), np.uint8)
    h_sc[...] = np.tile(base, (reps, 1))
    h_out = libecc_b200.pinned_empty((n, 2 * plen), np.uint8)
    h_st = libecc_b200.pinned_empty(n, np.int8)
    me = libecc_b200.MultiEngine(curve, devices=list(range(n_dev)), comb_window=DEFAULT_COMB.get(curve, 0))
    me.prj_pt_mul_batch(h_sc, None, out=h_out, status=h_st)          # warm-up (stage buffers, first-touch)
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        me.prj_pt_mul_batch(h_sc, None, out=h_out, status=h_st)
        times.append(time.perf_counter() - t0)
    want, wst = oracle_smul(curve, base[:128])
    ok = True
    for g in range(n_dev):                                            # first items of every device's shard
        lo = n * g // n_dev
        w, ws = oracle_smul(curve, h_sc[lo:lo + 64])
        ok = ok and bool((h_out[lo:lo + 64] == w).all() and (h_st[lo:lo + 64] == ws).all())
    me.close()
    best = min(times)
    return {"call": "eccb200_multi_prj_pt_mul_batch", "devices": n_dev, "items": n, "e2e_value": n / best, "unit": unit,
            "seconds_best_of_3": best, "seconds_all": times, "h2d_bytes": n * qlen, "d2h_bytes": n * (2 * plen + 1),
            "timing": "host wall clock around the blocking call (one process, one host thread per GPU)",
            "parity_first_items_of_every_shard": ok}


if __name__ == "__main__":
    main()
