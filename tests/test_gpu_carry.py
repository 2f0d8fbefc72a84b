"""The carry corpus (tests/carry_corpus.py) on the GPU: the rows that drive every carry of the device arithmetic both ways in the
CPU simulation (tests/test_carry.py) run through the compiled chains, via each op's host entry point and via fq_dev_run3 with
iters = 1, and every row must equal its reference (the C oracle where it has the op, else the Python oracle)."""
import numpy as np
import pytest

import carry_corpus

pytestmark = pytest.mark.gpu

OUT = {"decode": 64}                                  # output row bytes where they differ from the first input's
STATUS = ("decode", "dh_endo")


@pytest.fixture(scope="module")
def fq():
    import fourq_b200
    assert fourq_b200.device_count() >= 1        # raises if the CUDA library or device is missing: no silent fallback
    return fourq_b200


def _host(L, rs, out, st):
    """rs through its host entry point on one GPU."""
    lib, p = L.lib(), L.ptr
    ins = [p(x) for x in rs.ins]
    kind, _, name = rs.op.partition("_")
    n = rs.n
    if rs.op == "fp2_select":
        return lib.fq_fp2_select(ins[2], ins[0], ins[1], p(out), n, 1)
    if kind == "fp2":
        return getattr(lib, "fq_" + rs.op)(*ins, p(out), n, 1)
    if kind == "fp":
        return lib.fq_fp_op(L.FPOP[name], ins[0], ins[1] if len(ins) > 1 else None, p(out), n, 1)
    if kind == "f25519":
        return lib.fq_fp25519_op(L.FPOP[name], ins[0], ins[1] if len(ins) > 1 else None, p(out), n, 1)
    if rs.op in ("x25519", "mul_base", "mul_endo_base"):
        return getattr(lib, "fq_" + rs.op)(*ins, p(out), n, 1)
    if rs.op in ("decode", "dh_endo"):
        return getattr(lib, "fq_" + rs.op)(*ins, p(out), p(st), n, 1)
    raise AssertionError(rs.op)


def _device(fq, rs, width):
    """rs through fq_dev_run3 on GPU 0, iters = 1."""
    from fourq_b200 import device
    bufs = [device.DeviceBuffer.from_host(0, x) for x in rs.ins]
    out = device.DeviceBuffer(0, rs.n * width)
    st = device.DeviceBuffer(0, rs.n) if rs.op in STATUS else None
    try:
        a = bufs + [None] * (3 - len(bufs))
        device.dev_run(rs.op, 0, a[0], a[1], out, st, rs.n, iters=1, c=a[2])
        return out.to_host((rs.n, width)), (st.to_host((rs.n,)) if st is not None else None)
    finally:
        for b in bufs + [out, st]:
            if b is not None:
                b.free()


SETS = carry_corpus.build()


@pytest.mark.parametrize("rs", SETS, ids=[rs.name for rs in SETS])
def test_carry_corpus_on_the_gpu(fq, rs):
    from fourq_b200 import _lib as L
    want_out, want_st = carry_corpus.reference(rs)
    width = OUT.get(rs.op, rs.ins[0].shape[1] if rs.op not in ("mul_base", "mul_endo_base", "dh_endo") else 32)
    out = np.full((rs.n, width), 0xEE, np.uint8)
    st = np.full(rs.n, 0xEE, np.uint8) if rs.op in STATUS else None
    L.check(_host(L, rs, out, st))
    dev_out, dev_st = _device(fq, rs, width)
    for path, o, s in (("host", out, st), ("fq_dev_run3", dev_out, dev_st)):
        bad = np.flatnonzero(~(o == want_out).all(axis=1) | (False if want_st is None else s != want_st))
        assert not len(bad), (path, rs.name, len(bad), [bytes(x).hex() for x in rs.ins[0][bad[:3]]])
