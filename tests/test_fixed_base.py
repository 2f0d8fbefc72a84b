"""Fixed-base DH and scalar multiplication for a caller-registered point (fq_base_create, fq_dh_fixed, fq_mul_fixed) without a
GPU: the per-digit tables and the comb of comb.cuh in the CPU simulation (tests/hostsim/fixed_base_sim.cpp), against the C oracle
and against the plain affine group law of tests/torsion.py; then the host engine of capi.cu compiled against the mock CUDA
runtime with the mock kernels of tests/hostsim/mock_kernels_fixed.cpp (registration, lazy per-GPU tables, error paths, threads)."""
import ctypes
import hashlib
import os
import random
import subprocess
import threading

import numpy as np
import pytest

import torsion
from fourq_b200 import _lib
from oracle import c_oracle as C
from oracle import fourq_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_DIR = os.path.join(HERE, "hostsim")
N = O.N
P = _lib.ptr
COMB_WORDS = 63 * 8 * 24
# SHA-256 of the [2][12,096] words of the G and [392]G tables built at context creation, before the table construction took
# the base as a point: the tables must stay word for word the same
G_TABLES_SHA256 = "1a65a658de579d2ee459d105a8f31b27f0ffabb6148d9c0806567d154d4364fd"
EDGE = [0, 1, 2, N - 1, N, N + 1, 2 * N, (1 << 256) - 1]


def _stale(target):
    srcs = [os.path.join(SIM_DIR, f) for f in os.listdir(SIM_DIR) if f.endswith((".cpp", ".h", ".sh"))]
    csrc = os.path.join(HERE, "..", "fourq_b200", "csrc")
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h")) or f == "capi.cu"]
    return not os.path.exists(target) or os.path.getmtime(target) < max(os.path.getmtime(s) for s in srcs)


@pytest.fixture(scope="module")
def sim():
    so = os.path.join(SIM_DIR, "libfq_hostsim_fixed.so")
    if _stale(so) or _stale(os.path.join(SIM_DIR, "libfq_mockengine_fixed.so")):
        subprocess.check_call(["sh", os.path.join(SIM_DIR, "build_fixed_base.sh")])
    L = ctypes.CDLL(so)
    L.sim_comb_point.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t]
    L.sim_comb_tables.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    return L


@pytest.fixture(scope="module")
def eng(sim):
    L = _lib.bind(ctypes.CDLL(os.path.join(SIM_DIR, "libfq_mockengine_fixed.so")))
    L.mock_live_allocs.restype = ctypes.c_long
    L.mock_live_allocs.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_long)]
    L.mock_fail_nth.argtypes = [ctypes.c_char_p, ctypes.c_int]
    L.mock_violations.restype = ctypes.c_long
    L.mock_set_device_count(4)
    L.mock_set_jitter_us(0)
    yield L
    L.mock_set_jitter_us(0)


def rows(lst, width=32):
    return np.frombuffer(b"".join(lst), np.uint8).reshape(len(lst), width).copy()


def scal_rows(ks):
    return rows([int(k % (1 << 256)).to_bytes(32, "little") for k in ks])


def ref_r(k):
    """r of MUL_windowed (curve4q.py:216-219): k mod N, plus N if that is even."""
    r = k % N
    return r + N if r % 2 == 0 else r


def sim_tables(sim, xy):
    out = np.zeros(2 * COMB_WORDS, np.uint32)
    sim.sim_comb_tables(P(xy) if xy is not None else None, P(out))
    return out


def sim_fixed(sim, dh, xy, k):
    n = k.shape[0]
    out = np.full((n, 32), 0xEE, np.uint8); st = np.full(n, 9, np.uint8)
    xy = np.frombuffer(xy, np.uint8).copy() if isinstance(xy, bytes) else xy
    sim.sim_comb_point(dh, P(xy), P(k), P(out), P(st) if dh else None, n)
    return out, st


def test_g_tables_are_unchanged_and_registration_builds_the_same(sim):
    t0 = sim_tables(sim, None)
    assert hashlib.sha256(t0.tobytes()).hexdigest() == G_TABLES_SHA256
    genc = C.mul_base(scal_rows([1]))
    gxy, st = C.decode(genc)
    assert st[0] == 0
    assert (sim_tables(sim, gxy[0]) == t0).all()
    # a registered [392]G: the table of P = [392]G is the DH table of G, word for word (entries are canonical affine)
    qxy, st = C.decode(C.mul_base(scal_rows([392])))
    assert st[0] == 0
    assert (sim_tables(sim, qxy[0])[:COMB_WORDS] == t0[COMB_WORDS:]).all()


def _points_and_scalars():
    rng = random.Random(11)
    ks = EDGE + [rng.getrandbits(256) for _ in range(4)]
    return scal_rows(ks)


def test_dh_fixed_prime_order_points_against_the_oracle(sim):
    k = _points_and_scalars()
    n = k.shape[0]
    pts = [e for e, _ in torsion.prime_order_points(32)] + [bytes(C.mul_base(scal_rows([1]))[0])]
    for e in pts:
        xy, st = C.decode(rows([e]))
        assert st[0] == 0
        want, wst = C.dh(k, np.repeat(rows([e]), n, axis=0))
        out, ost = sim_fixed(sim, 1, xy[0], k)
        assert (ost == wst).all() and (out == want).all(), e.hex()


def test_dh_fixed_torsion_and_shifted_points_against_the_oracle(sim):
    """Every point of the 392-torsion subgroup and a prime-order point shifted by each: encoded registration where the point
    decodes (fq_dh on the broadcast encoding), affine registration for all (encode(DH_windowed(k, P)))."""
    k = _points_and_scalars()
    n = k.shape[0]
    A = torsion.prime_order_points(1, seed=3)[0][1]
    pts = [T for T, _ in torsion.torsion_points()] + [torsion.add(A, T) for T, _ in torsion.torsion_points()]
    for pt in pts:
        xy = np.frombuffer(torsion.xy(pt), np.uint8).copy()
        axy, ast = C.dh_affine(k, np.repeat(xy[None], n, axis=0))
        want = np.where((ast == 0)[:, None], C.encode(axy), 0)
        out, ost = sim_fixed(sim, 1, xy, k)
        assert (ost == ast).all() and (out == want).all(), pt
        e = torsion.enc(pt)
        dxy, dst = C.decode(rows([e]))
        if dst[0] == 0:
            assert (dxy[0] == xy).all()
            want, wst = C.dh(k, np.repeat(rows([e]), n, axis=0))
            assert (ost == wst).all() and (out == want).all(), pt
        if pt in [T for T, _ in torsion.torsion_points()]:
            assert (ost == 5).all() and not out.any()


def test_mul_fixed_is_mul_windowed_not_k_times_p(sim):
    """[r]P with the reference's r, for points with a small-order component too: checked against the plain affine group law,
    and on a sample against the oracle's MUL_windowed.  [k]P differs from it on such points, and the test says so."""
    tors = torsion.torsion_points()
    A = torsion.prime_order_points(1, seed=4)[0][1]
    by_order = {}
    for T, o in tors:
        by_order.setdefault(o, T)
    pts = [by_order[7], by_order[8], by_order[56], torsion.add(A, by_order[7]), torsion.add(A, by_order[8]), torsion.add(A, by_order[28]), A]
    rng = random.Random(12)
    ks = [1, 2, 3, 4, N - 1, N, N + 1, 2 * N, (1 << 256) - 1] + [rng.getrandbits(256) for _ in range(5)]
    k = scal_rows(ks)
    differs = 0
    for pt in pts:
        out, _ = sim_fixed(sim, 0, torsion.xy(pt), k)
        for i, m in enumerate(ks):
            want = torsion.enc(torsion.mul(ref_r(m), pt))
            assert bytes(out[i]) == want, (pt, m)
            differs += want != torsion.enc(torsion.mul(m, pt))
        for i in (0, 1, len(ks) - 1):
            R = O.r1_to_affine(O.mul_windowed(ks[i], O.affine_to_r1(*pt)))
            assert bytes(out[i]) == bytes(O.encode(*R)), (pt, ks[i])
    assert differs > 0


# ---------------------------------------------------------------- the host engine against the mock CUDA runtime

def _create(eng, pt, affine=0):
    st = np.full(1, 9, np.uint8)
    h = ctypes.c_void_p(1)
    rc = eng.fq_base_create(P(np.frombuffer(pt, np.uint8).copy()), affine, P(st), ctypes.byref(h))
    return rc, int(st[0]), h


def _good(eng, pt, affine=0):
    rc, st, h = _create(eng, pt, affine)
    assert rc == 0 and st == 0 and h.value, eng.fq_last_error()
    return h


def _dh(eng, h, k, ndev):
    n = k.shape[0]
    out = np.full((n, 32), 0xEE, np.uint8); st = np.full(n, 9, np.uint8)
    assert eng.fq_dh_fixed(h, P(k), P(out), P(st), n, ndev) == 0, eng.fq_last_error()
    return out, st


def _mul(eng, h, k, ndev):
    out = np.full((k.shape[0], 32), 0xEE, np.uint8)
    assert eng.fq_mul_fixed(h, P(k), P(out), k.shape[0], ndev) == 0, eng.fq_last_error()
    return out


def _dev_allocs(eng):
    return eng.mock_live_allocs(2, None)


def test_engine_registration_rejects_bad_points(eng):
    e = bytes(C.mul_base(scal_rows([5]))[0])
    bad = bytearray(e); bad[15] |= 0x80                                   # reserved bit
    nonc = bytearray(32); nonc[:16] = ((1 << 127) - 1).to_bytes(16, "little")   # y0 = p
    t0 = bytes(torsion.enc(torsion.NEUTRAL))                              # (0, 1): the reference's t == 0 quirk
    off = None
    for y in range(2, 200):                                               # an encoding that decodes to no point
        c = bytearray(32); c[0] = y
        if C.decode(rows([bytes(c)]))[1][0] == 4:
            off = bytes(c)
            break
    for pt, want in ((bytes(bad), 1), (bytes(nonc), 2), (t0, 3), (off, 4)):
        assert C.decode(rows([pt]))[1][0] == want
        rc, st, h = _create(eng, pt)
        assert (rc, st, h.value) == (0, want, None), eng.fq_last_error()
    xy = bytearray(torsion.xy(torsion.prime_order_points(1)[0][1])); xy[0] ^= 1
    rc, st, h = _create(eng, bytes(xy), 1)
    assert (rc, st, h.value) == (0, 4, None)
    # the affine points of order 1, 2 and 4 that decode rejects are valid affine registrations
    for T, o in torsion.torsion_points()[:4]:
        h = _good(eng, torsion.xy(T), 1)
        out, st = _dh(eng, h, scal_rows([1, 2, 3]), 1)
        assert (st == 5).all() and not out.any()
        assert eng.fq_base_destroy(h) == 0


def test_engine_null_arguments_and_no_device(eng):
    e = np.frombuffer(bytes(C.mul_base(scal_rows([5]))[0]), np.uint8).copy()
    st = np.zeros(1, np.uint8); h = ctypes.c_void_p()
    k = scal_rows([1, 2]); out = np.zeros((2, 32), np.uint8); s2 = np.zeros(2, np.uint8)
    assert eng.fq_base_create(None, 0, P(st), ctypes.byref(h)) == _lib.FQ_ERR_ARG
    assert eng.fq_base_create(P(e), 0, None, ctypes.byref(h)) == _lib.FQ_ERR_ARG
    assert eng.fq_base_create(P(e), 0, P(st), None) == _lib.FQ_ERR_ARG
    assert eng.fq_dh_fixed(None, P(k), P(out), P(s2), 2, 1) == _lib.FQ_ERR_ARG
    assert eng.fq_mul_fixed(None, P(k), P(out), 2, 1) == _lib.FQ_ERR_ARG
    assert eng.fq_base_dev_run(None, 1, 0, None, None, None, 2, 1, None) == _lib.FQ_ERR_ARG
    assert eng.fq_base_destroy(None) == 0
    h = _good(eng, bytes(e))
    assert eng.fq_dh_fixed(h, None, P(out), P(s2), 2, 1) == _lib.FQ_ERR_ARG
    assert eng.fq_dh_fixed(h, P(k), P(out), None, 2, 1) == _lib.FQ_ERR_ARG
    assert eng.fq_mul_fixed(h, P(k), None, 2, 1) == _lib.FQ_ERR_ARG
    assert eng.fq_mul_fixed(h, P(k), P(out), 2, 5) == _lib.FQ_ERR_ARG           # 4 mock devices
    assert eng.fq_dev_run(64, 0, P(k), None, P(out), P(s2), 2, 1, None) == _lib.FQ_ERR_ARG     # the internal op needs a base
    assert eng.fq_base_destroy(h) == 0
    eng.mock_set_device_count(0)
    try:
        assert eng.fq_base_create(P(e), 0, P(st), ctypes.byref(h)) == _lib.FQ_ERR_NO_DEVICE
    finally:
        eng.mock_set_device_count(4)


def _destroy_freed(eng, h):
    """fq_base_destroy, returning how many device buffers it freed (the handle's tables: one buffer per GPU it was used on)."""
    before = _dev_allocs(eng)
    assert eng.fq_base_destroy(h) == 0
    return before - _dev_allocs(eng)


def test_engine_lazy_tables_ndev_trim_and_dev_run(eng, sim):
    rng = np.random.default_rng(21)
    n = 1003
    k = rng.integers(0, 256, (n, 32), np.uint8)
    k[:len(EDGE)] = scal_rows(EDGE)
    A = torsion.prime_order_points(1, seed=9)[0][1]
    T8 = [T for T, o in torsion.torsion_points() if o == 8][0]
    xy = torsion.xy(torsion.add(A, T8))
    want_dh, want_st = sim_fixed(sim, 1, xy, k)
    want_mul, _ = sim_fixed(sim, 0, xy, k)
    for ndev in (1, 2, 3, 4):
        h = _good(eng, xy, 1)
        assert _destroy_freed(eng, _good(eng, xy, 1)) == 0                   # registration alone builds nothing
        out, st = _dh(eng, h, k, ndev)
        assert (out == want_dh).all() and (st == want_st).all(), ndev
        assert (_mul(eng, h, k, ndev) == want_mul).all(), ndev
        assert _destroy_freed(eng, h) == ndev                                # tables on the GPUs the calls used, and only there
    h = _good(eng, xy, 1)
    assert (_mul(eng, h, k, 4) == want_mul).all()
    assert eng.fq_trim() == 0
    out, st = _dh(eng, h, k, 4)                                               # the handle survives fq_trim
    assert (out == want_dh).all() and (st == want_st).all()
    # device-resident runs on the tables of the handle
    dk, dout, dst = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
    for p_, sz in ((dk, n * 32), (dout, n * 32), (dst, n)):
        assert eng.fq_dev_alloc(1, ctypes.byref(p_), sz) == 0
    assert eng.fq_dev_upload(1, dk, P(k), n * 32) == 0
    ms = ctypes.c_float()
    assert eng.fq_base_dev_run(h, 1, 1, dk, dout, dst, n, 2, ctypes.byref(ms)) == 0, eng.fq_last_error()
    got = np.zeros((n, 32), np.uint8); gst = np.zeros(n, np.uint8)
    assert eng.fq_dev_download(1, P(got), dout, n * 32) == 0 and eng.fq_dev_download(1, P(gst), dst, n) == 0
    assert (got == want_dh).all() and (gst == want_st).all()
    assert eng.fq_base_dev_run(h, 0, 1, dk, dout, None, n, 1, ctypes.byref(ms)) == 0
    assert eng.fq_dev_download(1, P(got), dout, n * 32) == 0 and (got == want_mul).all()
    for p_ in (dk, dout, dst):
        assert eng.fq_dev_free(1, p_) == 0
    assert _destroy_freed(eng, h) == 4
    assert eng.mock_violations() == 0


@pytest.mark.parametrize("api", [b"cudaMalloc", b"cudaStreamSynchronize"])
def test_engine_failed_table_build(eng, sim, api):
    k = scal_rows([1, 2, 3, N + 5])
    e = torsion.prime_order_points(1, seed=17)[0][0]
    warm = _good(eng, e)
    _dh(eng, warm, k, 1)                                                  # contexts and staging on GPU 0 exist
    assert eng.fq_base_destroy(warm) == 0
    h = _good(eng, e)
    before = _dev_allocs(eng)
    eng.mock_fail_nth(api, 1)                                             # the next call of `api` is the table build's
    out = np.zeros((4, 32), np.uint8); st = np.zeros(4, np.uint8)
    rc = eng.fq_dh_fixed(h, P(k), P(out), P(st), 4, 1)
    eng.mock_fail_nth(api, 0)
    assert rc == _lib.FQ_ERR_CUDA and eng.fq_last_error() != b""
    assert _dev_allocs(eng) == before                                     # nothing left allocated
    xy, _ = C.decode(rows([e]))
    want, wst = sim_fixed(sim, 1, xy[0], k)
    out, st = _dh(eng, h, k, 1)
    assert (out == want).all() and (st == wst).all()
    assert _dev_allocs(eng) == before + 1
    assert eng.fq_base_destroy(h) == 0 and _dev_allocs(eng) == before


def test_engine_threads_two_handles_four_gpus(eng, sim):
    eng.mock_set_jitter_us(100)
    rng = np.random.default_rng(23)
    n = 700
    pts = [torsion.xy(A) for _, A in torsion.prime_order_points(2, seed=29)]
    hs = [_good(eng, p, 1) for p in pts]
    ks = [rng.integers(0, 256, (n, 32), np.uint8) for _ in range(3)]
    want = {}
    for t in range(3):
        for b in range(2):
            want[t, b] = (sim_fixed(sim, 1, pts[b], ks[t]), sim_fixed(sim, 0, pts[b], ks[t])[0])
    errs = []

    def work(t):
        for it in range(3):
            b = (t + it) % 2
            ndev = 1 + (t + it) % 4
            out = np.zeros((n, 32), np.uint8); st = np.zeros(n, np.uint8); mo = np.zeros((n, 32), np.uint8)
            if eng.fq_dh_fixed(hs[b], P(ks[t]), P(out), P(st), n, ndev) or eng.fq_mul_fixed(hs[b], P(ks[t]), P(mo), n, ndev):
                errs.append((t, it, "rc"))
                continue
            (wo, wst), wm = want[t, b]
            if not ((out == wo).all() and (st == wst).all() and (mo == wm).all()):
                errs.append((t, it, b, ndev))
    try:
        ts = [threading.Thread(target=work, args=(t,)) for t in range(3)]
        [t.start() for t in ts]; [t.join() for t in ts]
    finally:
        eng.mock_set_jitter_us(0)
        for h in hs:
            assert eng.fq_base_destroy(h) == 0
    assert not errs and eng.mock_violations() == 0
