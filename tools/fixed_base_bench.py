#!/usr/bin/env python
"""Fixed-base DH and scalar multiplication for one registered point (fourq_b200.FixedBase) next to the paths a caller would
otherwise use, on one GPU; prints one JSON line.

    python tools/fixed_base_bench.py [--rows 16777216] [--e2e-rows 1048576] [--reps 5] [--dev 0]

  kernel        device-resident CUDA-event time of one launch on --rows rows (2^24 by default: 512 MiB of scalars, more than
                the 126 MB of L2; 256 MiB of zeros are written between timed launches), one warm-up launch each, the four
                operations alternating rep by rep in this process: dh_fixed and mul_fixed on the registered point, dh_endo
                (variable-base DH, the point broadcast to every row) and mul_base_comb (keygen on the tables of G)
  e2e           host entry points on --e2e-rows rows from page-locked (fourq_b200.pinned_empty) and from ordinary numpy
                arrays, best of --reps after one warm-up call
  registration  fq_base_create, and the first call on the device (n = 1, builds the tables) next to the second
Every timed output is compared with fourq_b200.DH on the same rows (point broadcast), and mul_fixed with MUL_base."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fourq_b200 as fq                                    # noqa: E402
from fourq_b200 import device as fqdev                     # noqa: E402


def gpu_info(dev):
    """name and power limit of the card, read now with nvidia-smi"""
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:          # the numbers still stand; say where the card information is missing
        return {"gpu": None, "power_limit": None, "gpu_info_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1 << 24)
    ap.add_argument("--e2e-rows", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dev", type=int, default=0)
    a = ap.parse_args()
    dev, n = a.dev, a.rows
    fq.set_device(dev)
    rng = np.random.default_rng(2024)
    enc = fq.MUL_base(rng.integers(0, 256, (1, 32), np.uint8))[0]          # a public key: the registered point

    # registration latency: create, then the first call on the device (builds the tables) and the second
    fq.DH(np.zeros((1, 32), np.uint8), enc[None].copy())                    # device context and engine threads exist already
    one = rng.integers(0, 256, (1, 32), np.uint8)
    t0 = time.perf_counter(); fb = fq.FixedBase(enc); t1 = time.perf_counter()
    fb.MUL(one); t2 = time.perf_counter()
    fb.MUL(one); t3 = time.perf_counter()
    reg = {"create_ms": (t1 - t0) * 1e3, "first_call_ms": (t2 - t1) * 1e3, "second_call_ms": (t3 - t2) * 1e3}

    # device-resident kernels
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = np.broadcast_to(enc, (n, 32)).copy()
    dk = fqdev.DeviceBuffer.from_host(dev, k); dp = fqdev.DeviceBuffer.from_host(dev, pub)
    outs = {op: (fqdev.DeviceBuffer(dev, n * 32), fqdev.DeviceBuffer(dev, n)) for op in ("dh_fixed", "mul_fixed", "dh_endo", "mul_base_comb")}

    def run(op):
        o, s = outs[op]
        if op == "dh_fixed":
            return fqdev.dev_run_fixed(fb, True, dev, dk, o, s, n)
        if op == "mul_fixed":
            return fqdev.dev_run_fixed(fb, False, dev, dk, o, None, n)
        if op == "dh_endo":
            return fqdev.dev_run("dh_endo", dev, dk, dp, o, s, n)
        return fqdev.dev_run("mul_base_comb", dev, dk, None, o, None, n)
    times = {op: [] for op in outs}
    for op in outs:
        run(op)                                                             # warm-up
    for _ in range(a.reps):
        for op in outs:
            fqdev.flush_l2(dev)
            times[op].append(run(op))
    want, wst = fq.DH(k, pub)
    match = {}
    for op in ("dh_fixed", "dh_endo"):
        o, s = outs[op]
        match[op] = bool((o.to_host((n, 32)) == want).all() and (s.to_host((n,)) == wst).all())
    match["mul_base_comb"] = bool((outs["mul_base_comb"][0].to_host((n, 32)) == fq.MUL_base(k)).all())
    mul_host = fb.MUL(k)
    match["mul_fixed"] = bool((outs["mul_fixed"][0].to_host((n, 32)) == mul_host).all())
    kernel = {op: {"best_ms": min(t), "median_ms": float(np.median(t)), "rows_per_s": n / (min(t) * 1e-3)} for op, t in times.items()}
    del dk, dp, outs

    # end to end, host arrays
    m = a.e2e_rows
    km = k[:m].copy()
    pk = fq.pinned_empty((m, 32)); pk[:] = km
    po = fq.pinned_empty((m, 32)); ps = fq.pinned_empty((m,))
    pp = fq.pinned_empty((m, 32)); pp[:] = pub[:m]
    o = np.zeros((m, 32), np.uint8); s = np.zeros(m, np.uint8)
    cases = {
        "dh_fixed_pinned": lambda: fb.DH(pk, out=po, status=ps),
        "dh_fixed_pageable": lambda: fb.DH(km, out=o, status=s),
        "mul_fixed_pinned": lambda: fb.MUL(pk, out=po),
        "mul_fixed_pageable": lambda: fb.MUL(km, out=o),
        "dh_endo_pinned": lambda: fq.DH(pk, pp, out=po, status=ps),
        "dh_endo_pageable": lambda: fq.DH(km, pub[:m], out=o, status=s),
    }
    e2e = {}
    for name, fn in cases.items():
        fn()
        best = 1e30
        for _ in range(a.reps):
            t = time.perf_counter(); fn(); best = min(best, time.perf_counter() - t)
        e2e[name] = {"best_ms": best * 1e3, "rows_per_s": m / best}
        res = (po if "pinned" in name else o)
        match["e2e_" + name] = bool((res == (want[:m] if name.startswith("dh") else mul_host[:m])).all())
    fb.close()
    print(json.dumps(dict(gpu_info(dev), rows=n, e2e_rows=m, reps=a.reps, kernel=kernel, e2e=e2e, registration=reg,
                          outputs_match=match, all_match=all(match.values()))))
    return 0 if all(match.values()) else 1


if __name__ == "__main__":
    sys.exit(main())
