#!/usr/bin/env python
"""The stream entry points (fourq_b200.cuda, fq_stream_run) next to the paths a caller would otherwise use, on one GPU;
prints one JSON line.

    python tools/stream_bench.py [--large 1048576,16777216] [--small 1024,16384] [--reps 5] [--dev 0]

  large   device-resident dh_endo and mul_base_comb on --large rows (inputs in GPU memory): fq_dev_run3 (one launch on the
          engine's own stream, its CUDA-event time) against fq_stream_run on a torch stream (CUDA events on that stream
          around the call: the kernels plus the pool allocation, the scratch wipe and its release), alternating rep by rep;
          256 MiB of zeros are written before each timed launch so that no input is read from L2.  Median of --reps.
  small   wall time per batch of --small DH rows (dh_endo) in three ways: the host entry point from page-locked arrays, one
          stream call plus a synchronisation of its stream, and the replay of a CUDA graph that captured that call plus a
          synchronisation.  Median over 200 batches after 20 warm-up batches.
Every path's output is compared with the host entry point on the same rows."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fourq_b200 as fq                                    # noqa: E402
import fourq_b200.cuda as fc                               # noqa: E402
from fourq_b200 import _lib                                # noqa: E402


def gpu_info(dev):
    """name and power limit of the card, read now with nvidia-smi"""
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:          # the numbers still stand; say where the card information is missing
        return {"gpu": None, "power_limit": None, "gpu_info_error": str(e)}


def inputs(n, seed, dev):
    """n scalars and n valid encoded points (a failing row every 4,096), made on the GPU by comb keygen"""
    rng = np.random.default_rng(seed)
    k = torch.from_numpy(rng.integers(0, 256, (n, 32), np.uint8)).cuda(dev)
    k2 = torch.from_numpy(rng.integers(0, 256, (n, 32), np.uint8)).cuda(dev)
    pub = fc.MUL_base(k2)
    pub[::4096] = 0xFF
    return k, pub


def large(n, reps, dev):
    L = _lib.lib()
    k, pub = inputs(n, 1, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:%d" % dev)
    s = torch.cuda.Stream(device=dev)
    res = {}
    for op, b, has_st in (("dh_endo", pub, True), ("mul_base_comb", None, False)):
        code = _lib.DEVOP[op]
        out_d = torch.empty((n, 32), dtype=torch.uint8, device="cuda:%d" % dev)
        out_s = torch.empty_like(out_d)
        st_d = torch.empty(n, dtype=torch.uint8, device="cuda:%d" % dev) if has_st else None
        st_s = torch.empty_like(st_d) if has_st else None
        p = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        ms = ctypes.c_float()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_dev, t_str = [], []
        for r in range(reps + 1):                                         # rep 0 warms both paths up
            torch.cuda.synchronize(dev)
            fq.device.flush_l2(dev)
            _lib.check(L.fq_dev_run3(code, dev, p(k), p(b), None, p(out_d), p(st_d), n, 1, ctypes.byref(ms)))
            with torch.cuda.stream(s):
                flush.zero_()
                e0.record(s)
                _lib.check(L.fq_stream_run(code, p(k), p(b), None, p(out_s), p(st_s), n, s.cuda_stream))
                e1.record(s)
            e1.synchronize()
            if r:
                t_dev.append(ms.value); t_str.append(e0.elapsed_time(e1))
        assert torch.equal(out_d, out_s) and (not has_st or torch.equal(st_d, st_s)), op
        md, mst = float(np.median(t_dev)), float(np.median(t_str))
        res[op] = {"dev_run_ms": md, "stream_ms": mst, "stream_minus_dev_run_ms": mst - md,
                   "dev_run_Mrows_s": n / md / 1e3, "stream_Mrows_s": n / mst / 1e3}
        del out_d, out_s, st_d, st_s
    del k, pub, flush
    torch.cuda.empty_cache()
    return res


def small(n, dev, batches=200, warm=20):
    rng = np.random.default_rng(n)
    k = fq.pinned_empty((n, 32)); k[:] = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.pinned_empty((n, 32)); pub[:] = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
    out = fq.pinned_empty((n, 32)); st = fq.pinned_empty((n,))
    want = fq.DH(k, pub)
    dk, dpub = torch.from_numpy(np.asarray(k)).cuda(dev), torch.from_numpy(np.asarray(pub)).cuda(dev)
    s = torch.cuda.Stream(device=dev)

    def wall(fn):
        for _ in range(warm):
            fn()
        t = []
        for _ in range(batches):
            t0 = time.perf_counter(); fn(); t.append(time.perf_counter() - t0)
        return float(np.median(t)) * 1e6

    def host():
        fq.DH(k, pub, out=out, status=st)

    with torch.cuda.stream(s):
        so, sst = fc.DH(dk, dpub)
    s.synchronize()

    def stream():
        fc.DH(dk, dpub, out=so, status=sst, stream=s)
        s.synchronize()

    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        go, gst = fc.DH(dk, dpub)

    def replay():
        g.replay()
        torch.cuda.synchronize(dev)

    r = {"host_pinned_us": wall(host), "stream_us": wall(stream), "graph_replay_us": wall(replay)}
    assert (np.asarray(out) == want[0]).all() and (so.cpu().numpy() == want[0]).all() and (go.cpu().numpy() == want[0]).all()
    assert (sst.cpu().numpy() == want[1]).all() and (gst.cpu().numpy() == want[1]).all()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--large", default="1048576,16777216")
    ap.add_argument("--small", default="1024,16384")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--dev", type=int, default=0)
    a = ap.parse_args()
    torch.cuda.set_device(a.dev)
    fq.set_device(a.dev)
    res = {"card": gpu_info(a.dev), "large": {}, "small": {}}
    for n in [int(x) for x in a.large.split(",") if x]:
        res["large"][n] = large(n, a.reps, a.dev)
    for n in [int(x) for x in a.small.split(",") if x]:
        res["small"][n] = small(n, a.dev)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
