"""GPU tests of the stream entry points (fq_stream_run, fq_base_stream_run) through the PyTorch adapter fourq_b200.cuda.

Every operation of test_gpu_shapes.OPS (each op of the host engine plus FixedBase.DH / .MUL) runs on CUDA tensors at
1, 127-129, 1,023-1,025 and a ragged ~100k rows, at COMB_TWO_WAVES +- 1 for the comb ops and at 2^22 + 1 rows for the
launch-group ops.  Bytes and statuses must equal the host entry point on the same rows, the rows past n must keep their
poison, and a sample must equal the oracle.  Then: ordering with torch work on the same stream, a call that returns while
its stream is still busy, two streams on two threads next to a host call, CUDA graph capture and replay, and the
refusals on real memory."""
import threading
import time

import numpy as np
import pytest

from test_gpu_shapes import COMB_TWO_WAVES, LAUNCH_GROUP, OPS, POISON, _first_diff, _host, _inputs, fixed_base, fq, pool  # noqa: F401

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

TAIL = 512
SAMPLE = 1500                     # random rows per op compared with the oracle, plus both ends of every size


@pytest.fixture(scope="module")
def fc(fq):
    import fourq_b200.cuda as fc
    assert torch.cuda.is_available()
    return fc


def _sizes(op):
    s = {1, 127, 128, 129, 1023, 1024, 1025, 100_003}
    if op.comb:
        s |= {COMB_TWO_WAVES - 1, COMB_TWO_WAVES + 1}
    if op.group:
        s.add(LAUNCH_GROUP + 1)
    return sorted(s)


def _stream_call(fc, op, ins, out, st, n, base):
    """The adapter function of op on the first n rows of the device inputs, into the given (poisoned) outputs."""
    a = [x[:n] for x in ins]
    o = out[:n]
    s = st[:n] if st is not None else None
    name = op.name
    if op.fixed == "dh":
        return fc.DH_fixed(base, a[0], out=o, status=s)
    if op.fixed == "mul":
        return fc.MUL_fixed(base, a[0], out=o)
    if name in ("dh", "dh_endo"):
        return fc.DH(a[0], a[1], out=o, status=s, algorithm="endo" if name == "dh_endo" else "windowed")
    if name in ("dh_affine", "dh_endo_affine"):
        return (fc.DH_endo if name == "dh_endo_affine" else fc.DH_windowed)(a[0], a[1], out=o, status=s)
    if name in ("dh_base", "dh_endo_base", "dh_base_comb"):
        return fc.DH_base(a[0], out=o, status=s, algorithm={"dh_base": "windowed", "dh_endo_base": "endo", "dh_base_comb": "comb"}[name])
    if name in ("mul_base", "mul_endo_base", "mul_base_comb"):
        return fc.MUL_base(a[0], out=o, algorithm={"mul_base": "windowed", "mul_endo_base": "endo", "mul_base_comb": "comb"}[name])
    if name in ("decode", "decode_spec"):
        return fc.decode(a[0], out=o, status=s, spec=name == "decode_spec")
    if name == "encode":
        return fc.encode(a[0], out=o)
    if name == "on_curve":
        return fc.PointOnCurve(a[0])
    if name == "x25519":
        return fc.x25519(a[0], a[1], out=o)
    if name.endswith("select"):
        return fc.run(name, a[0], a[1], a[2], out=o)
    return fc.run(name, *a, out=o)


@pytest.mark.parametrize("name", sorted(OPS))
def test_every_op_equals_the_host_path_and_the_oracle(fc, pool, fixed_base, name):  # noqa: F811
    op = OPS[name]
    sizes = _sizes(op)
    nmax = sizes[-1]
    ins = [x[:nmax] for x in _inputs(op, max(nmax, op.sizes()[-1]), pool)]     # _inputs plants hard rows up to op.sizes()
    rng = np.random.default_rng(len(name))
    rows = np.unique(np.concatenate([rng.integers(0, n, SAMPLE // len(sizes) + 1) for n in sizes] + [[0, n - 1] for n in sizes]))
    want_out, want_st = op.ref([x[rows] for x in ins])
    want_out = want_out.reshape(len(rows), op.out)
    dins = [torch.from_numpy(x).cuda() for x in ins]
    dout = torch.full((nmax + TAIL, op.out), POISON, dtype=torch.uint8, device="cuda")
    dst = torch.full((nmax + TAIL,), POISON, dtype=torch.uint8, device="cuda") if op.status else None
    for n in sizes:
        what = "%s n=%d" % (name, n)
        dout.fill_(POISON)
        if dst is not None:
            dst.fill_(POISON)
        res = _stream_call(fc, op, dins, dout, dst, n, fixed_base)
        torch.cuda.synchronize()
        if name == "on_curve":                          # PointOnCurve returns a new (N,) bool tensor
            got = res.cpu().numpy().astype(np.uint8)[:, None]
        else:
            got = dout.cpu().numpy()
            assert (got[n:] == POISON).all(), what + ": rows past n were written"
            got = got[:n]
        st = dst.cpu().numpy() if dst is not None else None
        if st is not None:
            assert (st[n:] == POISON).all(), what + ": statuses past n were written"
            st = st[:n]
        hout, hst = _host(op, [x[:n] for x in ins], n, 1, fixed_base)
        _first_diff(got, hout, what + ": stream vs host")
        if op.status:
            _first_diff(st[:, None], hst[:, None], what + ": stream vs host statuses")
        sel = rows < n
        _first_diff(got[rows[sel]], want_out[sel], what + ": stream vs oracle")
        if op.status:
            _first_diff(st[rows[sel], None], want_st[sel, None], what + ": stream vs oracle statuses")
    del dins, dout, dst
    torch.cuda.empty_cache()


# ---------------------------------------------------------------- ordering

def _dh_inputs(fq, n, seed):
    rng = np.random.default_rng(seed)
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
    pub[1] = 0xFF
    return k, pub


def test_inputs_made_by_torch_on_the_same_stream_just_before(fq, fc):
    n = 50_000
    k, pub = _dh_inputs(fq, n, 1)
    want = fq.DH(k ^ 0x5A, pub)
    s = torch.cuda.Stream()
    src = torch.from_numpy(k).cuda()
    dpub = torch.from_numpy(pub).cuda()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        kk = src ^ 0x5A                                   # a torch kernel on s writes the scalars ...
        out, st = fc.DH(kk, dpub)                         # ... and the DH call on s reads them, with no synchronisation
    s.synchronize()
    assert (out.cpu().numpy() == want[0]).all() and (st.cpu().numpy() == want[1]).all()


def _sleep_cycles(seconds):
    """GPU clock cycles of torch.cuda._sleep that take about `seconds` on this GPU (calibrated with events)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c = 20_000_000
    e0.record(); torch.cuda._sleep(c); e1.record(); e1.synchronize()
    return int(c * seconds * 1000.0 / max(e0.elapsed_time(e1), 1e-3))


def test_call_returns_while_the_stream_is_busy(fq, fc):
    n = 20_000
    k, pub = _dh_inputs(fq, n, 2)
    want = fq.DH(k, pub)
    dk, dpub = torch.from_numpy(k).cuda(), torch.from_numpy(pub).cuda()
    fc.DH(dk, dpub)                                       # the first call on the GPU initialises it
    torch.cuda.synchronize()
    cycles = _sleep_cycles(0.2)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(cycles)
        t0 = time.perf_counter()
        out, st = fc.DH(dk, dpub)
        dt = time.perf_counter() - t0
    busy = not s.query()
    s.synchronize()
    assert dt < 0.05, "the call took %.3f s behind a 0.2 s sleep" % dt
    assert busy, "the stream had finished when the call returned"
    assert (out.cpu().numpy() == want[0]).all() and (st.cpu().numpy() == want[1]).all()


# ---------------------------------------------------------------- concurrency

def test_two_streams_two_threads_and_a_host_call(fq, fc):
    jobs = [_dh_inputs(fq, 70_000 + 1000 * i, 10 + i) for i in range(3)]
    wants = [fq.DH(k, p) for k, p in jobs]
    res, errs = {}, []

    def stream_thread(i):
        try:
            k, p = jobs[i]
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                dk, dp = torch.from_numpy(k).cuda(non_blocking=False), torch.from_numpy(p).cuda()
                for _ in range(3):
                    out, st = fc.DH(dk, dp, stream=s)
            s.synchronize()
            res[i] = (out.cpu().numpy(), st.cpu().numpy())
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    def host_thread():
        try:
            k, p = jobs[2]
            res[2] = fq.DH(k, p)
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    ts = [threading.Thread(target=stream_thread, args=(i,)) for i in range(2)] + [threading.Thread(target=host_thread)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs
    for i in range(3):
        assert (res[i][0] == wants[i][0]).all() and (res[i][1] == wants[i][1]).all(), i


# ---------------------------------------------------------------- graphs

def test_graph_capture_and_replay(fq, fc, fixed_base):  # noqa: F811
    n = 30_000
    k, pub = _dh_inputs(fq, n, 20)
    sk, spub = torch.from_numpy(k).cuda(), torch.from_numpy(pub).cuda()
    sk2 = torch.from_numpy(k[::-1].copy()).cuda()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                         # warm-up outside capture: initialises the GPU and the base's tables
        fc.DH(sk, spub, algorithm="endo"); fc.DH_fixed(fixed_base, sk2); fc.decode(spub)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        dh_out, dh_st = fc.DH(sk, spub, algorithm="endo")
        fx_out, fx_st = fc.DH_fixed(fixed_base, sk2)
        xy, dst = fc.decode(spub)
    for rep in range(3):
        k, pub = _dh_inputs(fq, n, 30 + rep)
        k2 = np.random.default_rng(40 + rep).integers(0, 256, (n, 32), np.uint8)
        sk.copy_(torch.from_numpy(k)); spub.copy_(torch.from_numpy(pub)); sk2.copy_(torch.from_numpy(k2))
        g.replay()
        torch.cuda.synchronize()
        w = fq.DH(k, pub, algorithm="endo")
        assert (dh_out.cpu().numpy() == w[0]).all() and (dh_st.cpu().numpy() == w[1]).all(), rep
        w = fixed_base.DH(k2)
        assert (fx_out.cpu().numpy() == w[0]).all() and (fx_st.cpu().numpy() == w[1]).all(), rep
        w = fq.decode(pub)
        assert (xy.cpu().numpy() == w[0]).all() and (dst.cpu().numpy() == w[1]).all(), rep
    del g


# ---------------------------------------------------------------- refusals on real memory

def test_refusals_on_real_memory(fq, fc):
    from fourq_b200 import _lib
    n = 4096
    rng = np.random.default_rng(9)
    a = torch.from_numpy(rng.integers(0, 256, (n + 4, 32), np.uint8)).cuda()
    b = torch.from_numpy(rng.integers(0, 256, (n, 32), np.uint8)).cuda()
    out = torch.full((n, 32), POISON, dtype=torch.uint8, device="cuda")
    keep = a.clone()
    with pytest.raises(TypeError):
        fc.run("fp2_mul", a[:n].cpu(), b.cpu())
    L = _lib.lib()
    host = np.zeros((n, 32), np.uint8)
    s = torch.cuda.current_stream().cuda_stream
    assert L.fq_stream_run(_lib.DEVOP["fp2_mul"], _lib.ptr(host), b.data_ptr(), None, out.data_ptr(), None, n, s) == _lib.FQ_ERR_ARG
    flat = a.view(-1)
    off16 = flat[16:16 + 32 * n].view(n, 32)              # contiguous, but 16 bytes off the 32-byte rows
    with pytest.raises(fq.FourQError, match="aligned"):
        fc.run("fp2_mul", off16, b, out=out)
    with pytest.raises(fq.FourQError, match="alias"):
        fc.run("fp2_inv", a[:n], out=a[:n])
    partial = flat[32:32 + 32 * n].view(n, 32)            # out starts one row into a
    with pytest.raises(fq.FourQError, match="overlaps"):
        fc.run("fp2_mul", a[:n], b, out=partial)
    torch.cuda.synchronize()
    assert (out == POISON).all() and (a == keep).all()


def test_second_gpu_refusals_and_the_current_device(fq, fc):
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU: the cross-device cases need two")
    n = 1000
    rng = np.random.default_rng(10)
    a0 = torch.from_numpy(rng.integers(0, 256, (n, 32), np.uint8)).to("cuda:0")
    a1 = torch.from_numpy(rng.integers(0, 256, (n, 32), np.uint8)).to("cuda:1")
    out0 = torch.full((n, 32), POISON, dtype=torch.uint8, device="cuda:0")
    with pytest.raises(fq.FourQError, match="device"):
        fc.run("fp2_mul", a0, a1, out=out0)
    with pytest.raises(fq.FourQError, match="stream"):
        fc.run("fp2_mul", a0, a0, out=out0, stream=torch.cuda.Stream(device="cuda:1"))
    torch.cuda.synchronize(0)
    assert (out0 == POISON).all()
    torch.cuda.set_device(0)
    r = fc.run("fp2_mul", a1, a1)
    assert torch.cuda.current_device() == 0
    torch.cuda.synchronize(1)
    assert (r.cpu().numpy() == fq.GFp2.mul(a1.cpu().numpy(), a1.cpu().numpy())).all()
