#!/usr/bin/env python
"""End-to-end DH rate with page-locked vs ordinary (pageable) numpy arrays, in the combinations a caller can produce.
    [FQ_TRACE=1] python tools/pageable_check.py"""
import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fourq_b200 as fq
n = 1 << 20
rng = np.random.default_rng(1)
k = rng.integers(0, 256, (n, 32), np.uint8)
pub = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
pk = fq.pinned_empty((n, 32)); pk[:] = k
pp = fq.pinned_empty((n, 32)); pp[:] = pub
po = fq.pinned_empty((n, 32)); ps = fq.pinned_empty((n,))
o = np.zeros((n, 32), np.uint8); s = np.zeros((n,), np.uint8)
cases = (("pinned in/out", (pk, pp), dict(out=po, status=ps)), ("pageable in, fresh out", (k, pub), {}),
         ("pageable in, reused pageable out", (k, pub), dict(out=o, status=s)), ("pageable in, pinned out", (k, pub), dict(out=po, status=ps)),
         ("pinned in, fresh out", (pk, pp), {}), ("pinned in, reused pageable out", (pk, pp), dict(out=o, status=s)))
for name, args, kw in cases:
    for _ in range(2): fq.DH(*args, **kw)
    ts = []
    for _ in range(7):
        t = time.perf_counter(); fq.DH(*args, **kw); ts.append(time.perf_counter() - t)
    dt = float(np.median(ts))
    print("%-34s median %.2f ms  best %.2f ms  %.1f M rows/s" % (name, dt * 1e3, min(ts) * 1e3, n / dt / 1e6), flush=True)
