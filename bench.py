#!/usr/bin/env python
"""bench.py -- headline benchmark of fourq_b200: Curve4Q scalar multiplications per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...     (N > 1, one rank per GPU)

Workload (config.workload): BASELINE.json configs[2] -- variable-base DH, 2^20 (scalar, encoded point) rows per GPU:
decode + validate + cofactor clearing + scalar multiplication + inversion + encode, three kernel launches per step
(k_dh_prep -> k_dh_ladder -> k_dh_finish).  Every row is independent, so N GPUs run N independent slices (weak scaling, no collective on the data path;
torch.distributed is used only for the barrier and the max-over-ranks of the timings).

One JSON line is printed by rank 0:
  value      rows/s with inputs resident in HBM, CUDA-event time of the kernel, L2 flushed between steps
  e2e        the same rows through the public API fourq_b200.DH() from pinned host numpy arrays (H2D + kernels + D2H)
  roofline   dominant kernel k_dh_ladder: rows x algorithmic 32x32->64 multiply-adds of the main loop / its CUDA-event time,
             against the IMAD.WIDE.U32 issue peak measured live on the same GPU; roofline.step is the same for the whole
             step (SURVEY.md 8d "tight" count of decode + DH + encode: 58,284 endo / 103,836 windowed per row)
  cpu_baseline  the oracle (Python restatement of the reference) on the host's cores over a bounded sample; the same
             sample is compared bit-for-bit with the GPU output
  configs    (rank 0, after the timed regions, bounded): BASELINE cfg 2 (2^26 fp2 mul / sqr against the HBM peak, 2^20 inv), cfg 4
             (2^24 fixed-base keygen), cfg 5 (2^20 X25519 and its ratio to Curve4Q DH), kernel time with device-resident data
  e2e_pageable  the e2e call with plain numpy arrays (what a drop-in user passes); the engine stages them through pinned buffers
  inproc     (N > 1 only) rank 0 alone drives all N GPUs through the C ABI's own slice dispatcher (ndev = N) while the other
             ranks wait on a CPU barrier: cfg 4 strong scaling (2^24 rows at ndev 1 and N) and cfg 3 (N x 2^20 rows), each
             compared byte for byte with the ndev = 1 result
--impl reference times the reference's CPU algorithm (the oracle port: the reference itself is Python 2 and cannot run
here) with multiprocessing on all host cores, on a bounded sample per step.

--dump-outputs DIR writes what rank 0's last timed step of `value` returned, on a fixed sample of DUMP_ROWS rows (the same
rows in every run with the same --rows): DIR/out.npy (rows x 32 bytes of the encoded shared secret, float32), DIR/status.npy
(float32) and DIR/rows.npy (the sampled row indices, float64), 35 MiB in all.  The inputs are seeded, so two builds can be
compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "curve4q_variable_base_dh_scalar_mults_per_s"
UNIT = "scalar-mults/s"
ROWS_PER_GPU = 1 << 20
# SURVEY.md 8d, tight counts of 32x32->64 multiply-adds per row of cfg 3 for the algorithm that is run ...
IMADS_PER_ROW = {"windowed": 103836, "endo": 58284}
# ... and the share of the dominant kernel k_dh_ladder (the main loop): 62 x (4 DBL + ADD) / 64 x (DBL + ADD), DBL = 272, ADD = 384
IMADS_PER_ROW_LADDER = {"windowed": 62 * (4 * 272 + 384), "endo": 64 * (272 + 384)}
# the finish kernel shares one GF(p^2) inversion (1,504 multiply-adds, SURVEY 8d) between 16 rows at the price of 3 multiplications
# per row, so the step executes fewer multiply-adds than the reference's one-inversion-per-row count: the cheaper figure is cited
INV_ROWS = 16
INV_SAVING = 1504 - (1504 // INV_ROWS + 3 * 48)
# ... and the prepare kernel shares work the reference repeats: decode's two curve tests reuse y^2, d y^2 and x^2 (1 S + 2 M instead of
# 4 S + 4 M: 192 multiply-adds), and tau(P) is evaluated once for phi(P) and psi(P) (3 S + 5 M = 336, endomorphism path only)
PREP_SAVING = {"windowed": 192, "endo": 192 + 336}
BYTES_PER_ROW = 96              # 32 scalar + 32 point + 32 out
WORKLOAD = "cfg3 variable-base DH (decode+validate+[392]P+[k]Q+inversion+encode), 2^20 (scalar, encoded point) rows per GPU"
DUMP_ROWS = 1 << 18             # --dump-outputs sample: 2^18 x 33 float32 + 2^18 float64 = 35 MiB


def shard_bounds(n, world, rank):
    """Contiguous slice [lo, hi) of n rows owned by `rank` (same rule as the C ABI: ceil(n/world) rows per slice)."""
    per = (n + world - 1) // world
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def make_inputs(fq, rows, rank):
    """Seeded synthetic inputs (SURVEY.md 8d cfg 3): uniform scalars; public keys = [k']G for uniform k' (valid points)."""
    k = np.random.default_rng(3 + 1000 * rank).integers(0, 256, (rows, 32), np.uint8)
    kp = np.random.default_rng(4 + 1000 * rank).integers(0, 256, (rows, 32), np.uint8)
    pub = fq.MUL_base(kp)
    return k, pub


def dump_outputs(path, out, status):
    """Writes a fixed, seeded sample of DUMP_ROWS rows of one step's outputs (all rows when there are fewer) as float32 .npy
    files, with the sampled row indices."""
    rows = len(status)
    idx = np.arange(rows) if rows <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(rows, DUMP_ROWS, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "out.npy"), out[idx].astype(np.float32))
    np.save(os.path.join(path, "status.npy"), status[idx].astype(np.float32))
    np.save(os.path.join(path, "rows.npy"), idx.astype(np.float64))


class ClockSampler:
    """SM clock and throttle reasons of one GPU sampled every 10 ms (NVML, in-process) while the timed region runs;
    falls back to an `nvidia-smi -lms 100` child process when pynvml is not importable."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines = gpu, None, []
        self.nvml, self.handle, self.stop_flag, self.thread = None, None, False, None
        self.sm, self.mx, self.reasons = [], [], set()
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates all GPUs of the box; CUDA_VISIBLE_DEVICES may remap, so resolve through the PCI bus id when possible
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index(pynvml, gpu))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    @staticmethod
    def _nvml_index(pynvml, gpu):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [x.strip() for x in vis.split(",") if x.strip() != ""]
        if ids and all(x.isdigit() for x in ids) and gpu < len(ids):
            return int(ids[gpu])
        return gpu

    def _poll(self):
        n = self.nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
                self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
                r = int(get_reasons(self.handle))
                for nm, b in bits.items():
                    if r & b:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "samples": len(self.sm), "reasons": sorted(self.reasons), "source": "nvml, 10 ms period, during the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 100"}


# ---------------------------------------------------------------- CPU arm (oracle port of the reference)

def _cpu_row(args):
    from oracle import fourq_oracle as O
    return O.row_dh(args[0], args[1], mul=O.mul_endo if args[2] == "endo" else O.mul_windowed)


def cpu_dh(k, pub, procs, algorithm):
    """decode -> DH_windowed | DH_endo -> encode (the same reference algorithm as the GPU arm) on `procs` host processes."""
    import multiprocessing as mp
    with mp.get_context("fork").Pool(procs) as pool:
        t0 = time.perf_counter()
        res = pool.map(_cpu_row, [(bytes(k[i]), bytes(pub[i]), algorithm) for i in range(len(k))], chunksize=max(1, len(k) // (procs * 8)))
        dt = time.perf_counter() - t0
    return res, dt


def run_reference(args, rank, out):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host cores, bounded sample per step."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = 128 * cores
    # inputs for the CPU arm are generated on the CPU (valid points from the oracle's own fixed-base multiplication)
    from oracle import fourq_oracle as O
    rng = np.random.default_rng(3)
    k = rng.integers(0, 256, (sample, 32), np.uint8)
    base = [O.row_mul_base(bytes(r)) for r in np.random.default_rng(4).integers(0, 256, (16, 32), np.uint8)]
    pub = np.frombuffer(b"".join(base[i % 16] for i in range(sample)), np.uint8).reshape(sample, 32)
    for _ in range(args.warmup):
        cpu_dh(k[: 8 * cores], pub[: 8 * cores], cores, args.algorithm)
    total = 0.0
    for _ in range(args.steps):
        _, dt = cpu_dh(k, pub, cores, args.algorithm)
        total += dt
    value = sample * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "python-int", "data": "synthetic",
            "config": {"workload": WORKLOAD, "algorithm": "DH_%s" % args.algorithm, "sample_rows_per_step": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d rows per step x %d steps, oracle/fourq_oracle.py row_dh (DH_%s) under multiprocessing" % (sample, args.steps, args.algorithm)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), file=out, flush=True)


# ---------------------------------------------------------------- GPU arm

def _quiet_stdout():
    """Points fd 1 at stderr for the rest of the run (NCCL and other libraries print banners to stdout) and returns a file
    on the original stdout, so that the JSON line is the only thing the caller's stdout ever sees."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def _best_ms(fqdev, op, dev, a, b, out, st, n, reps=3, warm=1):
    for _ in range(warm):
        fqdev.dev_run(op, dev, a, b, out, st, n)
    best = 1e30
    for _ in range(reps):
        fqdev.flush_l2(dev)
        best = min(best, fqdev.dev_run(op, dev, a, b, out, st, n))
    return best


def measure_configs(fq, fqdev, dev, wide_peak, hbm, dh_ms, algorithm, quick=False):
    """BASELINE configs 2, 4 and 5 on one GPU, kernel time with device-resident inputs (CUDA events, best of 3, L2 flushed),
    each batch spot-checked against the oracle before it is reported.  About 1 s of GPU time plus the set-up of the arrays."""
    from oracle import fourq_oracle as O
    out = {}
    # ---- cfg 2: 2^26 mul / sqr (HBM-bound: 96 / 64 B per element), 2^20 inv (multiplier-bound)
    n = 1 << (20 if quick else 26)
    base = np.random.default_rng(2).integers(0, 256, (1 << 20, 32), np.uint8)
    a = np.tile(base, (n >> 20, 1)); b = np.tile(base[::-1], (n >> 20, 1))
    da = fqdev.DeviceBuffer.from_host(dev, a); db = fqdev.DeviceBuffer.from_host(dev, b); do = fqdev.DeviceBuffer(dev, n * 32)
    c2 = {"rows": n}
    for op, nbytes in (("fp2_mul", 96), ("fp2_sqr", 64)):
        ms = _best_ms(fqdev, op, dev, da, db if op == "fp2_mul" else None, do, None, n)
        got = do.to_host((128, 32))
        for j in range(128):
            assert bytes(got[j]) == O.row_fp2(op[4:], bytes(a[j]), bytes(b[j]) if op == "fp2_mul" else None), (op, j)
        c2[op + "_ms"] = ms; c2[op + "_gbs"] = n * nbytes / ms / 1e6; c2[op + "_frac_hbm"] = n * nbytes / ms / 1e6 / hbm
    ni = 1 << 20
    ms = _best_ms(fqdev, "fp2_inv", dev, da, None, do, None, ni)
    got = do.to_host((64, 32))
    for j in range(64):
        assert bytes(got[j]) == O.row_fp2("inv", bytes(a[j])), j
    inv_imads = 1504 // INV_ROWS + 3 * 48
    c2.update({"fp2_inv_rows": ni, "fp2_inv_ms": ms, "fp2_inv_per_s": ni / ms * 1e3, "fp2_inv_imads_per_row": inv_imads,
               "fp2_inv_frac_imad": ni * inv_imads / ms * 1e3 / wide_peak, "hbm_peak_gbs": hbm})
    out["cfg2"] = c2
    del da, db, do, a, b
    # ---- cfg 4: 2^24 fixed-base keygen [k]G on per-digit tables
    n = 1 << (20 if quick else 24)
    k = np.random.default_rng(5).integers(0, 256, (n, 32), np.uint8)
    dk = fqdev.DeviceBuffer.from_host(dev, k); do = fqdev.DeviceBuffer(dev, n * 32)
    ms = _best_ms(fqdev, "mul_base_comb", dev, dk, None, do, None, n)
    got = do.to_host((2048, 32))
    for j in range(0, 2048, 64):
        assert bytes(got[j]) == O.row_mul_base(bytes(k[j])), j
    comb_imads = 62 * 336 + 1504 // INV_ROWS + 5 * 48
    out["cfg4"] = {"rows": n, "kernel_ms": ms, "rows_per_s": n / ms * 1e3, "imads_per_row": comb_imads, "frac_imad": n * comb_imads / ms * 1e3 / wide_peak,
                   "algorithm": "per-digit tables: 62 mixed additions, no doubling (comb.cuh)"}
    del dk, do
    # ---- cfg 5: 2^20 X25519 next to 2^20 Curve4Q DH (the batched compare.py)
    n = 1 << 20
    kk = np.random.default_rng(6).integers(0, 256, (n, 32), np.uint8); uu = np.random.default_rng(7).integers(0, 256, (n, 32), np.uint8)
    dk = fqdev.DeviceBuffer.from_host(dev, kk); du = fqdev.DeviceBuffer.from_host(dev, uu); do = fqdev.DeviceBuffer(dev, n * 32); ds = fqdev.DeviceBuffer(dev, n)
    ms_x = _best_ms(fqdev, "x25519", dev, dk, du, do, None, n, reps=2)
    got = do.to_host((32, 32))
    for j in range(32):
        assert bytes(got[j]) == O.x25519(bytes(kk[j]), bytes(uu[j])), j
    pub = fq.MUL_base(np.random.default_rng(4).integers(0, 256, (n, 32), np.uint8))
    dp = fqdev.DeviceBuffer.from_host(dev, pub)
    other = "windowed" if algorithm == "endo" else "endo"
    ms_other = _best_ms(fqdev, "dh" if other == "windowed" else "dh_endo", dev, dk, dp, do, ds, n, reps=2)
    ms_alg = {algorithm: dh_ms, other: ms_other}
    out["cfg5"] = {"rows": n, "x25519_ms": ms_x, "x25519_rows_per_s": n / ms_x * 1e3, "dh_endo_ms": ms_alg["endo"], "dh_windowed_ms": ms_alg["windowed"],
                   "ratio_endo": ms_x / ms_alg["endo"], "ratio_windowed": ms_x / ms_alg["windowed"],
                   "x25519_frac_imad": n * 123078 / ms_x * 1e3 / wide_peak,
                   "note": "Curve4Q DH throughput / X25519 throughput; the draft claims >2x with endomorphisms, 1.2-1.6x without (draft-ladd-cfrg-4q.md:170-171)"}
    return out


def measure_inproc(fq, world, algorithm, quick=False):
    """Rank 0 alone, all `world` GPUs in ONE process through the C ABI's slice dispatcher (capi.cu: one feeder and one drainer
    thread per GPU): cfg 4 strong scaling (2^24 keygen rows at ndev = 1 and ndev = world) and cfg 3 (world x 2^20 DH rows),
    page-locked host arrays, wall clock, best of 3; every multi-GPU result is compared byte for byte with the ndev = 1 result."""
    res = {"n_gpus": world}
    fq.set_device(0)
    from fourq_b200 import _lib
    res["gpu_numa_nodes"] = [int(_lib.lib().fq_device_numa_node(i)) for i in range(world)]
    n4 = 1 << (20 if quick else 24)
    # arrays laid out for `world` GPUs: each GPU's slice of rows sits on that GPU's NUMA node where the platform allows it
    pk = fq.pinned_empty((n4, 32), ndev=world); pk[:] = np.random.default_rng(5).integers(0, 256, (n4, 32), np.uint8)
    po1 = fq.pinned_empty((n4, 32), ndev=world); poN = fq.pinned_empty((n4, 32), ndev=world)

    def best(fn, reps=3):
        fn()
        t = 1e30
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); t = min(t, time.perf_counter() - t0)
        return t
    t1 = best(lambda: fq.MUL_base(pk, out=po1, ndev=1))
    tN = best(lambda: fq.MUL_base(pk, out=poN, ndev=world))
    kN = fq.last_kernel_ms()
    from fourq_b200 import device as fqdev
    rows4 = fqdev.last_rows_per_device(world)          # the engine cuts later calls' slices by each GPU's measured speed, and idle GPUs steal
    same4 = bool((po1 == poN).all())
    res["cfg4"] = {"rows": n4, "ndev1_rows_per_s": n4 / t1, "ndevN_rows_per_s": n4 / tN, "ndev1_ms": t1 * 1e3, "ndevN_ms": tN * 1e3, "speedup": t1 / tN,
                   "ndevN_max_device_span_ms": kN, "ndevN_rows_per_device": rows4, "scaling": "strong", "parity_vs_ndev1": same4}
    # what the box can move: the same 64 B of host traffic per row with next to no arithmetic (GFp2.neg), ndev = 1 and ndev = world
    from fourq_b200 import _lib as L
    tc1 = best(lambda: L.check(L.lib().fq_fp2_neg(L.ptr(pk), L.ptr(po1), n4, 1)))
    tcN = best(lambda: L.check(L.lib().fq_fp2_neg(L.ptr(pk), L.ptr(po1), n4, world)))
    res["copy_probe"] = {"rows": n4, "bytes_per_row": 64, "ndev1_ms": tc1 * 1e3, "ndevN_ms": tcN * 1e3, "ndev1_host_gbs": n4 * 64 / tc1 / 1e9, "ndevN_host_gbs": n4 * 64 / tcN / 1e9,
                         "note": "fq_fp2_neg on the cfg 4 arrays: 32 B in + 32 B out per row and a trivial kernel -- the floor that host <-> device traffic puts under the cfg 4 call at the same ndev"}
    rows = (1 << (18 if quick else 20))
    n3 = rows * world
    k3 = fq.pinned_empty((n3, 32), ndev=world); k3[:] = np.random.default_rng(3).integers(0, 256, (n3, 32), np.uint8)
    p3 = fq.pinned_empty((n3, 32), ndev=world); p3[:] = poN[:n3] if n3 <= n4 else np.tile(poN, ((n3 + n4 - 1) // n4, 1))[:n3]
    o3 = fq.pinned_empty((n3, 32), ndev=world); s3 = fq.pinned_empty((n3,), ndev=world)
    tN3 = best(lambda: fq.DH(k3, p3, out=o3, status=s3, ndev=world, algorithm=algorithm))
    rows3 = fqdev.last_rows_per_device(world)
    m = min(n3, 1 << 18)                                 # a slice that crosses the first slice boundary when world > 4; ndev = 1 on the same rows
    lo = max(0, rows - m // 2)
    o1, s1 = fq.DH(k3[lo:lo + m], p3[lo:lo + m], ndev=1, algorithm=algorithm)
    same3 = bool((o1 == o3[lo:lo + m]).all() and (s1 == s3[lo:lo + m]).all())
    res["cfg3"] = {"rows": n3, "rows_per_s": n3 / tN3, "ms": tN3 * 1e3, "rows_per_device": rows3, "scaling": "weak", "parity_vs_ndev1": same3, "parity_rows": int(m)}
    res["parity_vs_ndev1"] = same4 and same3
    res["note"] = ("one process drives all GPUs through fq_mul_base_comb / fq_dh_endo with ndev = %d (contiguous slices, per-device feeder and drainer "
                   "threads, no collective); pinned host arrays, wall clock of the whole call, best of 3" % world)
    if not res["parity_vs_ndev1"]:
        raise SystemExit("PARITY FAILURE: the ndev = %d result differs from ndev = 1" % world)
    return res



def main():
    sys.dont_write_bytecode = True      # the tree may be read-only, and a benchmark run leaves nothing behind in it
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=ROWS_PER_GPU, help="rows per GPU (default 2^20, the BASELINE size)")
    ap.add_argument("--algorithm", default="endo", choices=["windowed", "endo"],
                    help="scalar-multiplication algorithm of the reference: MUL_windowed or MUL_endo (same outputs)")
    ap.add_argument("--cpu-sample", type=int, default=-1, help="rows of the CPU baseline sample (default 256 per core; 0 = skip)")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg 2 / 4 / 5 measurements and the in-process multi-GPU phase")
    ap.add_argument("--quick", action="store_true", help="developer runs: small cfg 2 / 4 / in-process batches")
    ap.add_argument("--verify-rows", type=int, default=-1, help="rows of rank 0's batch compared bit for bit with the C oracle after the timed regions (default all; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of rank 0's outputs of the last timed step to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    out = _quiet_stdout()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, out)
        return
    args.warmup = max(args.warmup, 3)

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")       # CPU-side barrier: ranks that wait on it leave their GPU idle

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    import fourq_b200 as fq
    from fourq_b200 import device as fqdev
    fq.set_device(local_rank)
    rows = args.rows
    k, pub = make_inputs(fq, rows, rank)

    devop = "dh_endo" if args.algorithm == "endo" else "dh"
    imads = IMADS_PER_ROW[args.algorithm]
    # ---- device-resident arm: `value`
    dk = fqdev.DeviceBuffer.from_host(local_rank, k)
    dp = fqdev.DeviceBuffer.from_host(local_rank, pub)
    dout = fqdev.DeviceBuffer(local_rank, rows * 32)
    dst = fqdev.DeviceBuffer(local_rank, rows)
    for _ in range(args.warmup):
        fqdev.dev_run(devop, local_rank, dk, dp, dout, dst, rows)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t_wall0 = time.perf_counter()
    kernel_ms, phase_ms = [], []
    for _ in range(args.steps):
        fqdev.flush_l2(local_rank)                       # untimed: write 256 MiB > L2 between timed iterations
        kernel_ms.append(fqdev.dev_run(devop, local_rank, dk, dp, dout, dst, rows))   # CUDA events on the launch stream
        phase_ms.append(fqdev.last_phase_ms())           # the same step's three kernels, one event pair each
    barrier()
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    total_ms = max_over_ranks(sum(kernel_ms))
    value = world * rows * args.steps / (total_ms * 1e-3)
    out_dev = dout.to_host((rows, 32))
    st_dev = dst.to_host((rows,))

    # ---- end-to-end arm through the public API from pinned host memory: `e2e`
    pk = fq.pinned_empty((rows, 32)); pk[:] = k
    pp = fq.pinned_empty((rows, 32)); pp[:] = pub
    po = fq.pinned_empty((rows, 32)); ps = fq.pinned_empty((rows,))
    for _ in range(2):
        fq.DH(pk, pp, out=po, status=ps, algorithm=args.algorithm)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out_e2e, st_e2e = fq.DH(pk, pp, out=po, status=ps, algorithm=args.algorithm)   # H2D of k and pub, kernels, D2H of out and status: every step
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * rows * args.steps / e2e_s
    assert (out_e2e == out_dev).all() and (st_e2e == st_dev).all() and not st_dev.any()
    # the same call with plain (pageable) numpy arrays, outputs allocated by the call: what a drop-in user of the reference writes
    for _ in range(2):
        fq.DH(k, pub, algorithm=args.algorithm)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out_pg, st_pg = fq.DH(k, pub, algorithm=args.algorithm)
    barrier()
    pg_s = max_over_ranks(time.perf_counter() - t0)
    e2e_pageable = world * rows * args.steps / pg_s
    assert (out_pg == out_dev).all() and (st_pg == st_dev).all()

    # ---- in-process multi-GPU phase: rank 0 drives all GPUs, the other ranks wait on the CPU barrier with idle GPUs
    inproc = None
    if dist is not None and not args.no_configs:
        del dk, dp, dout, dst
        fq.trim()
        barrier()
        if rank == 0:
            try:
                inproc = measure_inproc(fq, world, args.algorithm, quick=args.quick)
            except Exception as e:                       # a parity failure is a SystemExit and still aborts the run; anything else must not cost the headline line
                inproc = {"error": "%s: %s" % (type(e).__name__, e)}
            fq.set_device(local_rank)
        dist.barrier(group=cpu_group)

    # ---- roofline denominator measured live + CPU baseline and parity on a sample (rank 0)
    line = None
    if rank == 0:
        wide_peak, imad_peak = fqdev.imad_peak(local_rank)
        imads_run = imads - INV_SAVING - PREP_SAVING[args.algorithm]  # the step as executed (the cheaper figure is the one cited)
        step_achieved = (value / world) * imads_run                  # all three kernels of a step
        ph = [sum(p[i] for p in phase_ms) / len(phase_ms) for i in range(3)]      # rank 0's average ms: prepare, ladder, finish
        ladder_achieved = rows * IMADS_PER_ROW_LADDER[args.algorithm] / (ph[1] * 1e-3)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm = peaks.get("hbm_gbs", 6650.0)
        traffic = None        # dram__bytes_read.sum + dram__bytes_write.sum of one ladder launch, from the committed ncu --set full capture
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("k_dh_ladder_%s_2p20_rows_bytes" % args.algorithm)
            if traffic is not None and rows != ROWS_PER_GPU:
                traffic = None
        except (OSError, ValueError):
            pass
        roofline = {"bound": "imad", "kernel": "k_dh_ladder", "achieved": ladder_achieved / 1e12, "peak": wide_peak / 1e12, "unit": "T IMAD.WIDE/s",
                    "frac": ladder_achieved / wide_peak, "traffic": traffic,
                    "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one k_dh_ladder launch from the committed ncu --set full capture (profiles/traffic.json), not re-measured in this run",
                    "frac_of_imad32_peak": ladder_achieved / imad_peak,
                    "kernel_ms": {"k_dh_prep": ph[0], "k_dh_ladder": ph[1], "k_dh_finish": ph[2]},
                    "step": {"achieved": step_achieved / 1e12, "frac": step_achieved / wide_peak, "frac_of_imad32_peak": step_achieved / imad_peak, "imads_per_row": imads_run,
                             "imads_per_row_reference_count": imads},
                    "hbm": {"achieved": (value / world) * (BYTES_PER_ROW + 2 * 1156) / 1e9, "peak": hbm, "unit": "GB/s",
                            "frac": (value / world) * (BYTES_PER_ROW + 2 * 1156) / 1e9 / hbm,
                            "note": "all three kernels: 96 B of inputs/outputs + 1,156 B of scratch written and read once per row; not the bound"},
                    "note": "per GPU; dominant kernel k_dh_ladder: achieved = rows x %d algorithmic 32x32->64 multiply-adds per row of the main loop "
                            "/ its CUDA-event time; step = all three kernels, rows/s x %d (SURVEY 8d tight count of decode + DH + encode, less what the engine saves: one inversion per 16 rows, shared subexpressions in decode and table_endo); peak = "
                            "IMAD.WIDE.U32 issue rate measured live by fq_imad_peak (32-bit IMAD measured %.2f T/s); HBM is not the bound: "
                            "%d B/row algorithmic + 2.3 KiB/row of scratch -> %.3f of %s %.1f GB/s" % (
                                IMADS_PER_ROW_LADDER[args.algorithm], imads_run, imad_peak / 1e12, BYTES_PER_ROW,
                                (value / world) * (BYTES_PER_ROW + 2 * 1156) / 1e9 / hbm, "measured" if peaks else "fallback", hbm)}
        cores = os.cpu_count() or 1
        sample = args.cpu_sample if args.cpu_sample >= 0 else 256 * cores
        cpu = None
        if sample > 0:
            sample = min(sample, rows)
            res, dt = cpu_dh(k[:sample], pub[:sample], cores, args.algorithm)
            got = [(bytes(out_dev[i]), int(st_dev[i])) for i in range(sample)]
            if got != res:
                raise SystemExit("PARITY FAILURE: GPU output differs from the oracle on the CPU-baseline sample")
            cpu = {"value": sample / dt, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "first %d rows of rank 0's batch, oracle row_dh (DH_%s) under multiprocessing (%d procs); bit-exact with the GPU rows" % (sample, args.algorithm, cores)}
        # every row of rank 0's batch against the C restatement of the reference (oracle/fourq_oracle.c), all host cores
        parity = None
        if args.verify_rows != 0:
            from oracle import c_oracle
            m = rows if args.verify_rows < 0 else min(rows, args.verify_rows)
            t0 = time.perf_counter()
            want, wst = c_oracle.dh(k[:m], pub[:m])
            if not ((want == out_dev[:m]).all() and (wst == st_dev[:m]).all()):
                raise SystemExit("PARITY FAILURE: GPU output differs from oracle/fourq_oracle.c")
            parity = {"rows_checked": int(m), "bit_exact": True, "checker": "oracle/fourq_oracle.c (DH_windowed restatement, pinned to the reference's golden vectors)",
                      "seconds": time.perf_counter() - t0}
            parity["checker_rows_per_s"] = m / parity["seconds"]      # the C port on all host cores (threads), for scale
        configs = None
        if not args.no_configs and rows == ROWS_PER_GPU and world == 1:      # N > 1 runs carry `inproc` instead
            try:
                configs = measure_configs(fq, fqdev, local_rank, wide_peak, hbm, sum(kernel_ms) / len(kernel_ms), args.algorithm, quick=args.quick)
            except AssertionError:
                raise SystemExit("PARITY FAILURE: a configs batch differs from the oracle")
            except Exception as e:
                configs = {"error": "%s: %s" % (type(e).__name__, e)}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32", "data": "synthetic",
                "config": {"workload": WORKLOAD, "algorithm": "MUL_%s (curve4q.py:%s)" % (args.algorithm, "405-442" if args.algorithm == "endo" else "188-235"),
                           "table_select": "strict scan" if fq.get_select_mode() else "masked loads", "rows_per_gpu": rows, "l2": "flushed (256 MiB memset) between timed iterations",
                           "timing": "CUDA events around the three kernels of each step (k_dh_prep, k_dh_ladder, k_dh_finish), summed over steps, max over ranks", "wall_s_timed_region": wall},
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 64 * rows, "d2h_bytes_per_step": 33 * rows,
                        "note": "fourq_b200.DH(k, B, out=, status=) on pinned numpy arrays (inputs and outputs), wall clock, per GPU bytes"},
                "e2e_pageable": {"value": e2e_pageable, "unit": UNIT, "frac_of_e2e": e2e_pageable / e2e_value,
                                 "note": "fourq_b200.DH(k, B) on plain numpy arrays, outputs allocated by the call; the engine stages pageable operands through pinned buffers on its own threads"},
                "gpu_launches": 3 * args.steps,
                "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "configs": configs, "inproc": inproc}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out_dev, st_dev)
    barrier()
    if dist is not None:
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), file=out, flush=True)


if __name__ == "__main__":
    main()
