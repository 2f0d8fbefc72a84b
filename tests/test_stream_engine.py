"""fq_stream_run / fq_base_stream_run (capi.cu) WITHOUT a GPU: capi.cu built against the mock CUDA runtime of tests/hostsim,
whose streams are threads and whose kernels are the CPU simulation of the device code, plus mock_cuda_stream.cpp, which adds
the pool and capture calls and counts synchronising calls, allocations, pool blocks and the work pushed to streams
(build_stream.sh).  Checks the refusals, the results against the host path, that a call
after the first one on a GPU neither synchronises nor allocates, that every pool block is zeroed on its stream before it is
freed, the first-call-under-capture rule, and (stream_stress.cpp under ThreadSanitizer) that a stream call does not wait for a
host call that holds the GPU's lock."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from fourq_b200 import _lib

HERE = os.path.dirname(os.path.abspath(__file__))
SIM_DIR = os.path.join(HERE, "hostsim")
CSRC = os.path.join(HERE, "..", "fourq_b200", "csrc")
ERR_ARG = _lib.FQ_ERR_ARG
D = _lib.DEVOP
POISON = 0xEE
TAIL = 64                     # rows past n in every output buffer, which must keep their poison


def _stale(target):
    srcs = [os.path.join(SIM_DIR, f) for f in os.listdir(SIM_DIR) if f.endswith((".cpp", ".h", ".sh"))]
    srcs += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")) or f == "capi.cu"]
    return not os.path.exists(target) or os.path.getmtime(target) < max(os.path.getmtime(s) for s in srcs)


def _load(so, script):
    if _stale(os.path.join(SIM_DIR, so)):
        subprocess.check_call(["sh", os.path.join(SIM_DIR, script)])
    L = _lib.bind(ctypes.CDLL(os.path.join(SIM_DIR, so)))
    L.mock_counter.restype, L.mock_counter.argtypes = ctypes.c_long, [ctypes.c_char_p]
    L.mock_violations.restype = ctypes.c_long
    L.mock_stream_create.restype, L.mock_stream_create.argtypes = ctypes.c_void_p, [ctypes.c_int]
    L.mock_stream_sync.argtypes = [ctypes.c_void_p]
    L.mock_set_capturing.argtypes = [ctypes.c_void_p, ctypes.c_int]
    L.mock_device_alloc.restype, L.mock_device_alloc.argtypes = ctypes.c_void_p, [ctypes.c_int, ctypes.c_size_t]
    L.mock_device_free.argtypes = [ctypes.c_void_p]
    L.mock_set_device_count(4)
    return L


@pytest.fixture(scope="module")
def eng():
    return _load("libfq_mockengine_stream.so", "build_stream.sh")


@pytest.fixture(scope="module")
def eng_fixed():
    return _load("libfq_mockengine_stream_fixed.so", "build_stream.sh")


class Buf:
    """Mock device memory of GPU `dev` (host memory the mock registers as device memory), viewed as a numpy array."""

    def __init__(self, L, dev, nbytes):
        self.L, self.nbytes = L, nbytes
        self.ptr = L.mock_device_alloc(dev, nbytes)
        assert self.ptr
        self.arr = np.frombuffer((ctypes.c_uint8 * nbytes).from_address(self.ptr), np.uint8)

    @classmethod
    def of(cls, L, dev, a):
        b = cls(L, dev, a.nbytes)
        b.arr[:] = a.reshape(-1)
        return b

    def at(self, off):
        return ctypes.c_void_p(self.ptr + off)


def counters(L):
    return {k: L.mock_counter(k.encode()) for k in ("syncs", "mallocs", "pool_allocs", "pool_frees", "pool_unzeroed", "enqueued")}


def rand(seed, n, w):
    return np.random.default_rng(seed).integers(0, 256, (n, w), np.uint8)


def keys_and_points(L, n, seed):
    k = rand(seed, n, 32)
    pub = np.empty_like(k)
    assert L.fq_mul_base_comb(_lib.ptr(rand(seed + 1, n, 32)), _lib.ptr(pub), n, 1) == 0
    pub[3] = 0xFF                                                    # failing rows: zero fill and a status
    return k, pub


# ---------------------------------------------------------------- refusals

def test_refusals_enqueue_nothing_and_leave_the_outputs_alone(eng):
    L = eng
    n = 256
    s0 = L.mock_stream_create(0)
    a = Buf.of(L, 0, rand(1, n, 32)); b = Buf.of(L, 0, rand(2, n, 32))
    a1 = Buf.of(L, 1, rand(1, n, 32))
    big = Buf(L, 0, (n + TAIL) * 64)
    out = Buf(L, 0, (n + TAIL) * 64); st = Buf(L, 0, n + TAIL)
    host = rand(3, n, 32)
    # one warm-up call so that device 0 is initialised: the refusals below must not be masked by the first-call work
    assert L.fq_stream_run(D["fp2_add"], a.at(0), b.at(0), None, out.at(0), None, n, s0) == 0, L.fq_last_error()
    L.mock_stream_sync(s0)
    cases = {
        "unknown op": (99, a.at(0), b.at(0), None, out.at(0), None, n, s0),
        "registered-base op code without a base": (64, a.at(0), None, None, out.at(0), st.at(0), n, s0),
        "null b": (D["dh_endo"], a.at(0), None, None, out.at(0), st.at(0), n, s0),
        "null status": (D["dh_endo"], a.at(0), b.at(0), None, out.at(0), None, n, s0),
        "null out": (D["fp2_mul"], a.at(0), b.at(0), None, None, None, n, s0),
        "host memory": (D["fp2_mul"], _lib.ptr(host), b.at(0), None, out.at(0), None, n, s0),
        "range runs past the allocation": (D["fp2_mul"], a.at(0), b.at(0), None, out.at(0), None, 1 << 36, s0),
        "operands on two GPUs": (D["fp2_mul"], a.at(0), a1.at(0), None, out.at(0), None, n, s0),
        "stream of another GPU": (D["fp2_mul"], a.at(0), b.at(0), None, out.at(0), None, n, L.mock_stream_create(1)),
        "misaligned 32-byte rows": (D["fp2_mul"], big.at(16), b.at(0), None, out.at(0), None, n, s0),
        "misaligned 64-byte rows": (D["encode"], big.at(16), None, None, out.at(0), None, n, s0),
        "misaligned output": (D["fp2_mul"], a.at(0), b.at(0), None, out.at(16), None, n, s0),
        "misaligned 16-byte rows": (D["fp_mul"], big.at(8), big.at(16 * n + 64), None, out.at(0), None, n, s0),
        "partial overlap": (D["fp2_mul"], a.at(0), b.at(0), None, a.at(32), None, n - 1, s0),
        "alias of another row width": (D["decode"], big.at(0), None, None, big.at(0), st.at(0), n, s0),
        "fp2_inv out is a": (D["fp2_inv"], a.at(0), None, None, a.at(0), None, n, s0),
        "f25519_inv out is a": (D["f25519_inv"], a.at(0), None, None, a.at(0), None, n, s0),
        "status inside out": (D["decode"], a.at(0), None, None, out.at(0), out.at(64 * 4), n, s0),
    }
    snap_a, snap_b, snap_big = a.arr.copy(), b.arr.copy(), big.arr.copy()
    for what, args in cases.items():
        out.arr[:] = POISON; st.arr[:] = POISON
        before = counters(L)
        assert L.fq_stream_run(*args) == ERR_ARG, what
        assert L.fq_last_error(), what
        assert counters(L) == before, what + ": something was enqueued or allocated"
        assert (out.arr == POISON).all() and (st.arr == POISON).all(), what
        assert (a.arr == snap_a).all() and (b.arr == snap_b).all() and (big.arr == snap_big).all(), what
    before = counters(L)
    assert L.fq_base_stream_run(None, 1, a.at(0), out.at(0), st.at(0), n, s0) == ERR_ARG
    assert L.fq_stream_run(D["dh_endo"], a.at(0), b.at(0), None, out.at(0), st.at(0), 0, s0) == 0      # n == 0: nothing to do
    assert counters(L) == before
    assert L.mock_violations() == 0


def test_allowed_aliases_and_alignments(eng):
    """Exact aliases of equal row width are accepted (not the inversions'), and 16-byte GF(p) rows need only 16 bytes."""
    L = eng
    n = 300
    s = L.mock_stream_create(0)
    x, y = rand(4, n, 32), rand(5, n, 32)
    want = np.empty_like(x)
    assert L.fq_fp2_mul(_lib.ptr(x), _lib.ptr(y), _lib.ptr(want), n, 1) == 0
    a = Buf.of(L, 0, x); b = Buf.of(L, 0, y)
    assert L.fq_stream_run(D["fp2_mul"], a.at(0), b.at(0), None, a.at(0), None, n, s) == 0, L.fq_last_error()
    L.mock_stream_sync(s)
    assert (a.arr.reshape(n, 32) == want).all()
    f = rand(6, 2 * n + 1, 16)
    wantf = np.empty((n, 16), np.uint8)
    assert L.fq_fp_op(_lib.FPOP["add"], _lib.ptr(f[1:n + 1]), _lib.ptr(f[n + 1:]), _lib.ptr(wantf), n, 1) == 0
    fb = Buf.of(L, 0, f); o = Buf(L, 0, n * 16)
    assert L.fq_stream_run(D["fp_add"], fb.at(16), fb.at(16 * (n + 1)), None, o.at(0), None, n, s) == 0, L.fq_last_error()
    L.mock_stream_sync(s)
    assert (o.arr.reshape(n, 16) == wantf).all()


# ---------------------------------------------------------------- results, scratch and the steady state

def _inputs(L, op, n):
    if op in ("dh_endo", "dh"):
        k, pub = keys_and_points(L, n, 11)
        return [k, pub], 32, True, lambda ins, o, s: getattr(L, "fq_" + op)(*map(_lib.ptr, ins), _lib.ptr(o), _lib.ptr(s), n, 1)
    if op in ("dh_base_comb", "dh_endo_base"):
        return [rand(12, n, 32)], 32, True, lambda ins, o, s: getattr(L, "fq_" + op)(_lib.ptr(ins[0]), _lib.ptr(o), _lib.ptr(s), n, 1)
    if op == "mul_base":
        return [rand(13, n, 32)], 32, False, lambda ins, o, s: L.fq_mul_base(_lib.ptr(ins[0]), _lib.ptr(o), n, 1)
    if op == "x25519":
        return [rand(14, n, 32), rand(15, n, 32)], 32, False, lambda ins, o, s: L.fq_x25519(*map(_lib.ptr, ins), _lib.ptr(o), n, 1)
    if op == "decode":
        _, pub = keys_and_points(L, n, 16)
        return [pub], 64, True, lambda ins, o, s: L.fq_decode(_lib.ptr(ins[0]), _lib.ptr(o), _lib.ptr(s), n, 1)
    assert op == "fp2_mul"
    return [rand(17, n, 32), rand(18, n, 32)], 32, False, lambda ins, o, s: L.fq_fp2_mul(*map(_lib.ptr, ins), _lib.ptr(o), n, 1)


@pytest.mark.parametrize("op", ["fp2_mul", "decode", "dh_endo", "dh_endo_base", "mul_base", "dh_base_comb", "x25519"])
def test_results_equal_the_host_path_with_no_sync_and_no_malloc_after_the_first_call(eng, op):
    """One op of each scratch kind (none, variable-base DH, fixed-base hand-over, X25519), on device 1."""
    L = eng
    n = 257
    ins, ow, has_st, host = _inputs(L, op, n)
    want = np.empty((n, ow), np.uint8); wst = np.empty(n, np.uint8)
    assert host(ins, want, wst) == 0, L.fq_last_error()
    s = L.mock_stream_create(1)
    bufs = [Buf.of(L, 1, x) for x in ins]
    out = Buf(L, 1, (n + TAIL) * ow); st = Buf(L, 1, n + TAIL)
    args = [b.at(0) for b in bufs] + [None] * (3 - len(bufs))
    for rep in range(3):
        out.arr[:] = POISON; st.arr[:] = POISON
        before = counters(L)
        assert L.fq_stream_run(D[op], *args, out.at(0), st.at(0) if has_st else None, n, s) == 0, L.fq_last_error()
        L.mock_stream_sync(s)
        after = counters(L)
        got = out.arr.reshape(n + TAIL, ow)
        assert (got[:n] == want).all(), (op, rep)
        assert (got[n:] == POISON).all() and (st.arr[n:] == POISON).all(), "rows past n were written"
        if has_st:
            assert (st.arr[:n] == wst).all()
        else:
            assert (st.arr == POISON).all()
        pools = after["pool_allocs"] - before["pool_allocs"]
        assert pools == (0 if op in ("fp2_mul", "decode") else 1), pools
        assert after["pool_frees"] - before["pool_frees"] == pools and after["pool_unzeroed"] == 0
        if rep > 0 or op != "fp2_mul":          # fp2_mul runs first on device 1: its first call initialises the GPU
            assert after["syncs"] == before["syncs"], "a stream call synchronised"
            assert after["mallocs"] == before["mallocs"], "a stream call allocated outside the pool"
    assert L.mock_violations() == 0


def test_fq_trim_trims_the_pool_and_the_calling_threads_device_is_restored(eng):
    L = eng
    n = 130
    s = L.mock_stream_create(1)
    k = Buf.of(L, 1, rand(20, n, 32)); out = Buf(L, 1, n * 32)
    L.mock_set_current_device(2)
    assert L.fq_stream_run(D["mul_base_comb"], k.at(0), None, None, out.at(0), None, n, s) == 0, L.fq_last_error()
    assert L.mock_current_device() == 2
    L.mock_stream_sync(s)
    t0 = L.mock_counter(b"pool_trims")
    assert L.fq_trim() == 0
    assert L.mock_counter(b"pool_trims") > t0
    assert L.fq_stream_run(D["mul_base_comb"], k.at(0), None, None, out.at(0), None, n, s) == 0, L.fq_last_error()
    L.mock_stream_sync(s)
    assert L.mock_counter(b"pool_unzeroed") == 0


# ---------------------------------------------------------------- capture

def test_first_call_under_capture_is_refused_then_accepted(eng):
    """Device 3 has seen no stream call: the first one needs initialisation, which a capturing stream cannot take."""
    L = eng
    n = 200
    s = L.mock_stream_create(3)
    k = Buf.of(L, 3, rand(21, n, 32)); out = Buf(L, 3, n * 32); st = Buf(L, 3, n)
    out.arr[:] = POISON
    L.mock_set_capturing(s, 1)
    before = counters(L)
    assert L.fq_stream_run(D["dh_base_comb"], k.at(0), None, None, out.at(0), st.at(0), n, s) == ERR_ARG
    assert b"outside capture" in L.fq_last_error()
    assert counters(L) == before and (out.arr == POISON).all()
    L.mock_set_capturing(s, 0)
    assert L.fq_stream_run(D["dh_base_comb"], k.at(0), None, None, out.at(0), st.at(0), n, s) == 0, L.fq_last_error()
    L.mock_stream_sync(s)
    first = out.arr.copy()
    out.arr[:] = POISON
    L.mock_set_capturing(s, 1)
    before = counters(L)
    assert L.fq_stream_run(D["dh_base_comb"], k.at(0), None, None, out.at(0), st.at(0), n, s) == 0, L.fq_last_error()
    L.mock_set_capturing(s, 0)
    L.mock_stream_sync(s)
    after = counters(L)
    assert (out.arr == first).all()
    assert after["syncs"] == before["syncs"] and after["mallocs"] == before["mallocs"]


def test_unbuilt_base_under_capture_is_refused_then_accepted(eng_fixed):
    L = eng_fixed
    n = 150
    G = np.empty((1, 32), np.uint8)
    assert L.fq_mul_base(_lib.ptr(np.full((1, 32), 7, np.uint8)), _lib.ptr(G), 1, 1) == 0
    h, st1 = ctypes.c_void_p(), np.zeros(1, np.uint8)
    assert L.fq_base_create(_lib.ptr(G), 0, _lib.ptr(st1), ctypes.byref(h)) == 0 and st1[0] == 0 and h.value
    s = L.mock_stream_create(2)
    k = rand(22, n, 32)
    want = np.empty_like(k); wst = np.empty(n, np.uint8)
    assert L.fq_dh_fixed(h, _lib.ptr(k), _lib.ptr(want), _lib.ptr(wst), n, 1) == 0      # tables on device 0 only
    kb = Buf.of(L, 2, k); out = Buf(L, 2, n * 32); st = Buf(L, 2, n)
    # device 2 initialised by a call without the base; the base's tables there are still to be built
    assert L.fq_stream_run(D["mul_base_comb"], kb.at(0), None, None, out.at(0), None, n, s) == 0, L.fq_last_error()
    L.mock_stream_sync(s)
    out.arr[:] = POISON
    L.mock_set_capturing(s, 1)
    before = counters(L)
    assert L.fq_base_stream_run(h, 1, kb.at(0), out.at(0), st.at(0), n, s) == ERR_ARG
    assert b"outside capture" in L.fq_last_error() and b"base" in L.fq_last_error()
    assert counters(L) == before and (out.arr == POISON).all()
    L.mock_set_capturing(s, 0)
    assert L.fq_base_stream_run(h, 1, kb.at(0), out.at(0), st.at(0), n, s) == 0, L.fq_last_error()
    L.mock_stream_sync(s)
    assert (out.arr.reshape(n, 32) == want).all() and (st.arr == wst).all()
    out.arr[:] = POISON
    L.mock_set_capturing(s, 1)
    assert L.fq_base_stream_run(h, 0, kb.at(0), out.at(0), None, n, s) == 0, L.fq_last_error()
    L.mock_set_capturing(s, 0)
    L.mock_stream_sync(s)
    wmul = np.empty_like(k)
    assert L.fq_mul_fixed(h, _lib.ptr(k), _lib.ptr(wmul), n, 1) == 0
    assert (out.arr.reshape(n, 32) == wmul).all()
    assert L.fq_base_destroy(h) == 0
    assert L.mock_violations() == 0


# ---------------------------------------------------------------- no lock shared with host calls (ThreadSanitizer)

def test_stream_stress_under_tsan():
    """stream_stress.cpp: a stream call on a GPU whose lock a long host call holds finishes enqueueing without waiting for it;
    stream calls from several threads and host calls on the same GPUs all give the simulation's results."""
    exe = os.path.join(SIM_DIR, "stream_stress_tsan")
    if _stale(exe):
        subprocess.check_call(["sh", os.path.join(SIM_DIR, "build_stream.sh")])
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=1 second_deadlock_stack=1")
    r = subprocess.run([exe], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "Sanitizer" not in r.stderr, r.stdout[-2000:] + r.stderr[-4000:]
    assert "stream_stress ok" in r.stdout


# ---------------------------------------------------------------- the PyTorch adapter without a GPU

def test_import_fourq_b200_does_not_import_torch():
    code = "import sys, fourq_b200; assert 'torch' not in sys.modules, 'torch imported'; print('ok')"
    r = subprocess.run([os.sys.executable, "-c", code], capture_output=True, text=True, cwd=os.path.join(HERE, ".."))
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_adapter_argument_validation():
    torch = pytest.importorskip("torch")
    import fourq_b200.cuda as fc
    with pytest.raises(TypeError):
        fc.DH(torch.zeros((4, 32), dtype=torch.int32), torch.zeros((4, 32), dtype=torch.uint8))
    with pytest.raises(ValueError):
        fc.decode(torch.zeros((4, 31), dtype=torch.uint8))
    with pytest.raises(TypeError, match="CUDA"):
        fc.encode(torch.zeros((4, 64), dtype=torch.uint8))              # host memory: the numpy facade is for that
    with pytest.raises(ValueError):
        fc.run("dh", torch.zeros((4, 32), dtype=torch.uint8))           # curve operations have their own functions
