"""GPU tests of the code around the arithmetic, for every operation of the host engine (capi.cu describe()) and for
FixedBase.DH / .MUL: the launch wrappers, their grid and stride arithmetic, the launch-group loops and the host pipeline's
chunking.  Each operation runs at sizes derived from its own geometry, through its host entry point on pageable arrays and
through fq_dev_run3 (the device-resident path bench.py times) with iters = 1 and 2 on poisoned output buffers.  Both
paths must give the same bytes and statuses on every row, must leave the rows past n untouched, and sampled rows must
equal the C oracle (or the Python oracle where the C one lacks the operation).

Inputs are prefixes of one seeded array per operation, so row i's expected output does not depend on the size; the
reference runs once per operation on the union of the rows sampled at all sizes."""
import ctypes
import multiprocessing as mp
import os
import zlib

import numpy as np
import pytest

import adversarial
from oracle import c_oracle as C
from oracle import fourq_oracle as O

pytestmark = pytest.mark.gpu

M = 1 << 20
DH_CHUNK = 148 * 2 * 128 * 12          # capi.cu kDhChunkRows: full pipeline chunk of the variable-base DH ops
COMB_CHUNK = 148 * 2 * 256 * 4         # capi.cu kCombChunkRows: full pipeline chunk of the comb ops
ROW_QUANT = 128                        # capi.cu kRowQuant: chunks of the ramp-down (and the staged DH half chunk) round to it
LAUNCH_GROUP = 1 << 22                 # kernels.h FQ_DH_MAX_BATCH: rows per launch group of fqk_dh, fqk_fixed_base, fqk_comb
INV_ROWS, INV_THREADS = 16, 64         # batchinv.cuh FQ_BATCHINV_ROWS rows per thread, 64-thread CTAs of the inversion kernels
INV_GROUP = INV_ROWS * INV_THREADS     # 1,024 rows: one CTA of full inversion groups; above it the row stride grows
COMB_TWO_WAVES = 148 * 16 * 256        # kernels_comb.cu: from 148 SMs x 16 tiles of 256 rows on, k_comb runs 4 CTAs per SM, not 2
TAIL = 512                             # rows past n in the device output buffers that must keep their poison
POISON = 0xEE
SAMPLE_ALL = 20_000                    # up to this size every row is compared with the oracle
EDGE = 512                             # rows compared at each end of every chunk and launch group
RANDOM_SAMPLE = 2000

P25519 = O.P25519
X25519_ORDER8 = [325606250916557431795983626356110631294008115727848805560023387167927233504,
                 39382357235489614581723060781553021112529911719440698176882885853963445705823]
FIXED_SCALAR = 0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF1234567890ABCDE    # FixedBase point P = [FIXED_SCALAR]G


@pytest.fixture(scope="module")
def fq():
    import fourq_b200
    assert fourq_b200.device_count() >= 1        # raises if the CUDA library or device is missing: no silent fallback
    return fourq_b200


@pytest.fixture(scope="module")
def fixed_base(fq):
    with fq.FixedBase(_fixed_point()) as fb:
        yield fb


def _fixed_point():
    return bytes(C.mul_base(_scalars([FIXED_SCALAR]))[0])


# ---------------------------------------------------------------- the operations

def _call(name, order, pre=lambda base: ()):
    """The host entry point `name` called as name(*pre(base), operands in `order`, n, ndev); a, b, c = inputs, o = out, s = status."""
    def run(ptrs, n, ndev, base):
        return getattr(_lib().lib(), name)(*pre(base), *[ptrs[k] for k in order], n, ndev)
    return run


def _lib():
    from fourq_b200 import _lib as L
    return L


class Op:
    def __init__(self, name, ins, out, status, chunk, host, ref, kind, cta=None, inv=False, group=False, var_dh=False, comb=False,
                 fixed=None):
        self.name, self.ins, self.out, self.status, self.chunk, self.host, self.ref, self.kind = name, ins, out, status, chunk, host, ref, kind
        self.cta, self.inv, self.group, self.var_dh, self.comb, self.fixed = cta, inv, group, var_dh, comb, fixed

    # the rows of a full chunk when the inputs are pageable: capi.cu run_host halves it for the variable-base DH ops
    def staged_chunk(self):
        return self.chunk // 2 // ROW_QUANT * ROW_QUANT if self.var_dh else self.chunk

    def sizes(self):
        units = [self.cta, INV_GROUP if self.inv else None, self.chunk, LAUNCH_GROUP if self.group else None,
                 COMB_TWO_WAVES if self.comb else None, self.staged_chunk() if self.var_dh else None]
        s = {1}
        for u in units:
            if u:
                s |= {u - 1, u, u + 1}
        # one ragged size of several units: past a launch group by 2^20 + 77 rows, otherwise 2 1/3 chunks (at most ~1.1 M rows)
        s.add(LAUNCH_GROUP + M + 77 if self.group else min(2 * self.chunk + self.chunk // 3 + 77, 1_100_077))
        return sorted(s)


def _fp2(op):
    unary = op in ("sqr", "inv", "neg", "conj", "invsqrt")
    ref = _py_ref("fp2_invsqrt") if op == "invsqrt" else (lambda ins, op=op: (C.fp2(op, *ins), None))
    return Op("fp2_" + op, (32,) if unary else (32, 32), 32, False, M // 4 if op in ("inv", "invsqrt") else M,
              _call("fq_fp2_" + op, "ao" if unary else "abo"), ref, "fp2_inv" if op == "inv" else "fp2",
              cta=None if op == "inv" else 256, inv=op == "inv")


def _fp(op):
    unary = op in ("sqr", "inv", "neg", "invsqrt")
    code = _lib().FPOP[op]
    return Op("fp_" + op, (16,) if unary else (16, 16), 16, False, M // 4 if op in ("inv", "invsqrt") else M,
              _call("fq_fp_op", "abo", lambda base, code=code: (code,)), lambda ins, op=op: (C.fp(op, *ins), None), "fp", cta=256)


def _f25(op):
    unary = op in ("sqr", "inv")
    code = _lib().FPOP[op]
    return Op("f25519_" + op, (32,) if unary else (32, 32), 32, False, M // 4 if op == "inv" else M,
              _call("fq_fp25519_op", "abo", lambda base, code=code: (code,)), _py_ref("f25519_" + op),
              "f25_inv" if op == "inv" else "f25", cta=None if op == "inv" else 256, inv=op == "inv")


def _dh_ref(ins):
    return C.dh(*ins)


def _dh_affine_ref(ins):
    return C.dh_affine(*ins)


def _mul_base_ref(ins):
    return C.mul_base(ins[0]), None


def _fixed_dh_ref(ins):
    return C.dh(ins[0], np.tile(np.frombuffer(_fixed_point(), np.uint8), (ins[0].shape[0], 1)))


def _fixed_mul_ref(ins):
    # MUL gives [r]P with r = k mod N (plus N if even); P has prime order, so that is [k mod N]P = [(k mod N) FIXED_SCALAR]G
    ks = [int.from_bytes(bytes(r), "little") % O.N * FIXED_SCALAR % O.N for r in ins[0]]
    return C.mul_base(_scalars(ks)), None


def _ops():
    ops = [_fp2(op) for op in ("mul", "sqr", "inv", "add", "sub", "neg", "conj", "invsqrt")]
    ops += [Op("fp2_select", (32, 32, 1), 32, False, M, _call("fq_fp2_select", "cabo"), _py_ref("select"), "sel", cta=256),
            Op("fp_select", (16, 16, 1), 16, False, M, _call("fq_fp_select", "cabo"), _py_ref("select"), "sel", cta=256)]
    ops += [_fp(op) for op in ("mul", "sqr", "inv", "add", "sub", "neg", "invsqrt")]
    ops += [Op("decode", (32,), 64, True, M // 4, _call("fq_decode", "aos"), lambda ins: C.decode(ins[0]), "enc", cta=256),
            Op("decode_spec", (32,), 64, True, M // 4, _call("fq_decode_spec", "aos"), _py_ref("decode_spec"), "enc", cta=256),
            Op("encode", (64,), 32, False, M, _call("fq_encode", "ao"), lambda ins: (C.encode(ins[0]), None), "xy", cta=256),
            Op("on_curve", (64,), 1, False, M, _call("fq_point_on_curve", "ao"),
               lambda ins: (C.on_curve(ins[0]).astype(np.uint8)[:, None], None), "xy", cta=256)]
    dh = dict(status=True, chunk=DH_CHUNK, cta=128, inv=True, group=True, var_dh=True)     # kernels.h FQ_DH_THREADS = 128
    ops += [Op("dh", (32, 32), 32, host=_call("fq_dh", "abos"), ref=_dh_ref, kind="dh", **dh),
            Op("dh_endo", (32, 32), 32, host=_call("fq_dh_endo", "abos"), ref=_dh_ref, kind="dh", **dh),
            Op("dh_affine", (32, 64), 64, host=_call("fq_dh_affine", "abos"), ref=_dh_affine_ref, kind="dh_affine", **dh),
            Op("dh_endo_affine", (32, 64), 64, host=_call("fq_dh_endo_affine", "abos"), ref=_dh_affine_ref, kind="dh_affine", **dh)]
    fb = dict(chunk=M // 8, cta=256, inv=True, group=True, kind="k")                     # k_fixed_base: 256-thread CTAs
    ops += [Op("dh_base", (32,), 32, True, host=_call("fq_dh_base", "aos"), ref=lambda ins: C.dh_base(ins[0]), **fb),
            Op("dh_endo_base", (32,), 32, True, host=_call("fq_dh_endo_base", "aos"), ref=lambda ins: C.dh_base(ins[0]), **fb),
            Op("mul_base", (32,), 32, False, host=_call("fq_mul_base", "ao"), ref=_mul_base_ref, **fb),
            Op("mul_endo_base", (32,), 32, False, host=_call("fq_mul_endo_base", "ao"), ref=_mul_base_ref, **fb)]
    cb = dict(chunk=COMB_CHUNK, cta=256, inv=True, group=True, comb=True, kind="k")        # k_comb: tiles of 256 rows
    ops += [Op("dh_base_comb", (32,), 32, True, host=_call("fq_dh_base_comb", "aos"), ref=lambda ins: C.dh_base(ins[0]), **cb),
            Op("mul_base_comb", (32,), 32, False, host=_call("fq_mul_base_comb", "ao"), ref=_mul_base_ref, **cb),
            Op("fixed_dh", (32,), 32, True, host=_call("fq_dh_fixed", "aos", lambda base: (base.handle,)), ref=_fixed_dh_ref, fixed="dh", **cb),
            Op("fixed_mul", (32,), 32, False, host=_call("fq_mul_fixed", "ao", lambda base: (base.handle,)), ref=_fixed_mul_ref,
               fixed="mul", **cb)]
    ops += [Op("x25519", (32, 32), 32, False, M // 8, _call("fq_x25519", "abo"), _py_ref("x25519"), "x25519", cta=128, inv=True)]
    ops += [_f25(op) for op in ("mul", "sqr", "inv", "add", "sub")]
    return {op.name: op for op in ops}


# ---------------------------------------------------------------- references

_PY = {
    "fp2_invsqrt": lambda a: O.row_fp2("invsqrt", a),
    "select": lambda x, y, c: O.row_select(c[0], x, y),
    "decode_spec": lambda e: O.row_decode(e, spec=True),
    "x25519": O.x25519,
    "f25519_mul": lambda a, b: O.row_f25519("mul", a, b), "f25519_add": lambda a, b: O.row_f25519("add", a, b),
    "f25519_sub": lambda a, b: O.row_f25519("sub", a, b), "f25519_sqr": lambda a: O.row_f25519("sqr", a),
    "f25519_inv": lambda a: O.row_f25519("inv", a),
}


def _py_row(args):
    return _PY[args[0]](*args[1:])


def _py_ref(key):
    """The Python oracle's row function _PY[key] over the rows, in a fork pool as test_gpu_parity does."""
    def ref(ins):
        rows = [(key,) + tuple(bytes(x[i]) for x in ins) for i in range(ins[0].shape[0])]
        with mp.get_context("fork").Pool(min(16, os.cpu_count() or 1)) as pool:
            got = pool.map(_py_row, rows, chunksize=64)
        if key.startswith("decode"):
            return _rows([o for o, _ in got]), np.array([s for _, s in got], np.uint8)
        return _rows(got), None
    return ref


def _rows(lst):
    return np.frombuffer(b"".join(lst), np.uint8).reshape(len(lst), -1).copy()


def _scalars(ms):
    return _rows([int(m % (1 << 256)).to_bytes(32, "little") for m in ms])


OPS = _ops()


def test_table_covers_every_device_op():
    """Every op code of fq_dev_run3 has an entry, plus the two FixedBase ops."""
    assert set(OPS) == set(_lib().DEVOP) | {"fixed_dh", "fixed_mul"}


# ---------------------------------------------------------------- inputs

def _group_rows(n):
    """Rows of the inversion kernels' threads on n rows (thread t owns rows t + j * stride, j < 16; batchinv.cuh): one row at
    each position j, each of a different thread, and all 16 rows of thread 1."""
    groups = -(-n // INV_ROWS)
    stride = INV_THREADS * -(-groups // INV_THREADS)
    rows = [(5 + 3 * j) % stride + j * stride for j in range(INV_ROWS)] + [1 + j * stride for j in range(INV_ROWS)]
    return [r for r in rows if r < n]


def _plant(ins, hard, op, sizes):
    """Writes the hard rows (one array per input) at the start and across every size's last row, then the first hard
    rows (the zeros / failures, cycled) at the inversion-group positions of every size."""
    n = ins[0].shape[0]
    h = hard[0].shape[0]
    for lo in [0] + [max(0, s - h // 2) for s in sizes]:
        m = min(h, n - lo)
        for x, y in zip(ins, hard):
            x[lo:lo + m] = y[:m]
    if op.inv:
        nz = op.zero_rows
        rows = [r for s in sizes for r in _group_rows(s)]
        for i, r in enumerate(rows):
            for x, y in zip(ins, hard):
                x[r] = y[i % nz]


def _le(v, width):
    return np.frombuffer(int(v).to_bytes(width, "little"), np.uint8)


def _u(vals, width=32):
    return np.stack([_le(v, width) for v in vals])


def _inputs(op, n, pool):
    """(inputs, hard rows) of op at n rows; op.zero_rows = how many leading hard rows are zeros / failures for the inversion groups."""
    rng = np.random.default_rng(zlib.crc32(op.name.encode()))
    rand = [rng.integers(0, 256, (n, w), np.uint8) for w in op.ins]
    p = O.P127
    op.zero_rows = 0
    if op.kind in ("fp2", "fp2_inv", "fp", "sel"):
        a, b = adversarial.fp2_grid()
        if op.kind == "fp2_inv":
            zeros = _u([0, p, p << 128, p | p << 128, (2 * p), (2 * p) | p << 128, (2 * p) << 128])
            a = np.concatenate([zeros, a]); op.zero_rows = len(zeros)
        if op.kind == "sel":
            c = np.array([0, 1, 1, 0, 2, 3, 0x80, 0xFF, 0x7F, 0xFE], np.uint8)
            c = np.resize(c, a.shape[0])[:, None]
            rand[2] = (rand[2] & 1) if op.name.startswith("fp2") else rand[2]      # mostly 0 / 1, but any byte for fp_select
            hard = [a[:, :op.ins[0]], b[:, :op.ins[0]], c]
        else:
            hard = [a[:, :op.ins[0]], b[:, :op.ins[0]]][:len(op.ins)]
    elif op.kind in ("f25", "f25_inv"):
        vals = [0, P25519, 2 * P25519, 1, 2, 19, P25519 - 1, P25519 + 1, 2 * P25519 + 1, (1 << 255) - 1, 1 << 255, (1 << 256) - 1,
                (1 << 255) + 18, int("ff" * 16 + "00" * 16, 16), int("00" * 16 + "ff" * 16, 16), 1 << 128, (1 << 64) - 1]
        pairs = [(x, y) for x in vals for y in vals]
        hard = [_u([x for x, _ in pairs]), _u([y for _, y in pairs])][:len(op.ins)]
        if op.kind == "f25_inv":
            op.zero_rows = 3                                               # 0, p, 2p: zero mod p
            hard = [_u(vals)]
    elif op.kind == "enc":
        k, enc = adversarial.grid()
        low = [O.encode(x, y) for x, y in (((0, 0), (1, 0)), ((0, 0), (p - 1, 0)), ((0, 1), (0, 0)), ((0, p - 1), (0, 0)))]
        noncanonical = _u([p, p << 128, (p << 128) | (1 << 255)])
        hard = [np.concatenate([_rows(low), noncanonical, np.unique(enc, axis=0)])]
        rand[0] = pool["enc"][rng.integers(0, len(pool["enc"]), n)]
        bad = rng.random(n) < 0.25
        rand[0][bad] = rng.integers(0, 256, (int(bad.sum()), 32), np.uint8)
    elif op.kind == "xy":
        xy = pool["xy"][:64].copy()
        flip = xy.copy(); flip[:, 7] ^= 1                                  # off the curve
        hard = [np.concatenate([_u([0, p, (1 << 128) - 1, p | p << 128 | p << 256 | p << 384], 64), xy, flip])]
        rand[0] = pool["xy"][rng.integers(0, len(pool["xy"]), n)]
        bad = rng.random(n) < 0.25
        rand[0][bad] = rng.integers(0, 256, (int(bad.sum()), 64), np.uint8)
    elif op.kind in ("dh", "dh_affine"):
        G = O.encode(O.GX, O.GY)
        quirk = O.encode((0, 0), (1, 0))
        fails_k = _scalars([0, O.N, 2 * O.N, 5, 7, 9])
        fails_p = _rows([G, G, G, quirk, b"\xff" * 32, bytes(15) + b"\x80" + bytes(16)])
        k, enc = adversarial.grid()
        hk, hp = np.concatenate([fails_k, k]), np.concatenate([fails_p, enc])
        op.zero_rows = len(fails_k)
        i = rng.integers(0, len(pool["enc"]), n)
        rand[1] = pool["enc"][i] if op.kind == "dh" else pool["xy"][i]
        bad = rng.random(n) < 0.06
        rand[1][bad] = rng.integers(0, 256, (int(bad.sum()), op.ins[1]), np.uint8)
        if op.kind == "dh_affine":
            xy, st = C.decode(hp)
            xy[st != 0] = rng.integers(0, 256, (int((st != 0).sum()), 64), np.uint8)     # failed decodes: arbitrary rows
            xy[len(fails_k)::3, 9] ^= 1                                                    # some valid points pushed off the curve
            hp = xy
        hard = [hk, hp]
    elif op.kind == "k":
        hard = [_scalars([0, O.N, 2 * O.N] + adversarial.special_scalars())]
        op.zero_rows = 3
    elif op.kind == "x25519":
        us = [0, P25519, 1 << 255, (1 << 255) | P25519] + X25519_ORDER8 + [1, 9, P25519 - 1, P25519 + 1, 2 * P25519, (1 << 255) - 1,
                                                                          (1 << 256) - 1, int("ffffffff00000000" * 4, 16)]
        ks = [0, 1, 8, 1 << 254, (1 << 255) - 1, (1 << 256) - 1, int("a5" * 32, 16)]
        op.zero_rows = 6                                                   # u = 0 mod p after masking bit 255, or of order 8
        hu = _u(us + [u for _ in ks for u in us])
        hk = np.concatenate([rng.integers(0, 256, (len(us), 32), np.uint8), _u([k for k in ks for _ in us])])
        hard = [hk, hu]
    else:
        raise AssertionError(op.kind)
    ins = rand
    _plant(ins, hard, op, op.sizes())
    return ins


@pytest.fixture(scope="module")
def pool():
    """Valid encodings (C oracle [k]G) and their affine coordinates, which the DH and codec inputs draw from."""
    k = np.random.default_rng(7).integers(0, 256, (1 << 14, 32), np.uint8)
    enc = C.mul_base(k)
    xy, st = C.decode(enc)
    assert not st.any()
    return {"enc": enc, "xy": xy}


# ---------------------------------------------------------------- which rows are compared with the oracle

def _host_cuts(n, full):
    """Ends of the chunks a one-GPU host call cuts n rows into (capi.cu CallWork::init / take with ndev = 1): ramp up from
    full / 8 (at least 16,384) by doubling, full chunks, ramp down by halves rounded to ROW_QUANT."""
    small = min(max(full // 8, 16384), full)
    ramp = n > 2 * small
    lo, taken, cuts = 0, 0, []
    while lo < n:
        left, sz = n - lo, full
        if ramp:
            sz = small
            for _ in range(taken):
                if sz >= full:
                    break
                sz = min(2 * sz, full)
        m = min(sz, left)
        if ramp and small < left <= 2 * m:
            m = min((left // 2 + ROW_QUANT - 1) // ROW_QUANT * ROW_QUANT, full, left)
        lo += m
        taken += 1
        cuts.append(lo)
    return cuts


def _sample(op, n):
    """Every row up to SAMPLE_ALL rows; otherwise the first and last EDGE rows of every host chunk (pageable and pinned
    schedules) and launch group, so both sides of each boundary, and RANDOM_SAMPLE random rows."""
    if n <= SAMPLE_ALL:
        return np.arange(n)
    cuts = set(_host_cuts(n, op.staged_chunk())) | set(_host_cuts(n, op.chunk)) | {0, n}
    if op.group:
        cuts |= set(range(LAUNCH_GROUP, n, LAUNCH_GROUP))
    cuts = sorted(cuts)
    parts = [np.random.default_rng(n).integers(0, n, RANDOM_SAMPLE)]
    for lo, hi in zip(cuts, cuts[1:]):
        parts += [np.arange(lo, min(hi, lo + EDGE)), np.arange(max(lo, hi - EDGE), hi)]
    return np.unique(np.concatenate(parts))


def _first_diff(got, want, what):
    bad = np.flatnonzero((got != want).reshape(got.shape[0], -1).any(axis=1))
    assert bad.size == 0, "%s: %d rows differ, first %d: got %s want %s" % (
        what, bad.size, bad[0], bytes(got[bad[0]]).hex(), bytes(want[bad[0]]).hex())


# ---------------------------------------------------------------- the two paths

def _host(op, ins, n, ndev, base, out=None, status=None):
    out = np.empty((n, op.out), np.uint8) if out is None else out
    status = (np.empty(n, np.uint8) if status is None else status) if op.status else None
    L = _lib()
    ptrs = {"a": L.ptr(ins[0]), "b": L.ptr(ins[1]) if len(ins) > 1 else None, "c": L.ptr(ins[2]) if len(ins) > 2 else None,
            "o": L.ptr(out), "s": L.ptr(status)}
    L.check(op.host(ptrs, n, ndev, base))
    return out, status


class _Dev:
    """Device buffers of op for up to nmax rows, outputs with TAIL spare rows."""

    def __init__(self, op, ins, nmax):
        from fourq_b200 import device
        self.op, self.device = op, device
        self.ins = [device.DeviceBuffer.from_host(0, x[:nmax]) for x in ins]
        self.out = device.DeviceBuffer(0, (nmax + TAIL) * op.out)
        self.st = device.DeviceBuffer(0, nmax + TAIL) if op.status else None
        self.poison = np.full((nmax + TAIL) * op.out, POISON, np.uint8)

    def run(self, n, iters, base):
        L, op = _lib(), self.op
        for buf, w in ((self.out, op.out), (self.st, 1)):
            if buf is not None:
                L.check(L.lib().fq_dev_upload(0, buf.ptr, L.ptr(self.poison), (n + TAIL) * w))
        a = self.ins + [None] * (3 - len(self.ins))
        if op.fixed:
            self.device.dev_run_fixed(base, op.fixed == "dh", 0, a[0], self.out, self.st, n, iters=iters)
        else:
            self.device.dev_run(op.name, 0, a[0], a[1], self.out, self.st, n, iters=iters, c=a[2])
        return self.out.to_host((n + TAIL, op.out)), (self.st.to_host((n + TAIL,)) if self.st is not None else None)

    def free(self):
        for b in self.ins + [self.out, self.st]:
            if b is not None:
                b.free()


@pytest.mark.parametrize("name", sorted(OPS))
def test_every_size_host_and_device_path_against_the_oracle(fq, pool, fixed_base, name):
    op = OPS[name]
    sizes = op.sizes()
    nmax = sizes[-1]
    ins = _inputs(op, nmax, pool)
    samples = {n: _sample(op, n) for n in sizes}
    rows = np.unique(np.concatenate(list(samples.values())))
    want_out, want_st = op.ref([x[rows] for x in ins])
    want_out = want_out.reshape(len(rows), op.out)
    if op.status:
        assert len(set(want_st.tolist())) > 1, "the inputs must contain failing rows"
    dev = _Dev(op, ins, nmax)
    try:
        for n in sizes:
            what = "%s n=%d" % (name, n)
            out, st = _host(op, [x[:n] for x in ins], n, 1, fixed_base)
            if n == op.chunk + 1:
                kept = out, st
            d1, s1 = dev.run(n, 1, fixed_base)
            d2, s2 = dev.run(n, 2, fixed_base)
            _first_diff(d2, d1, what + ": dev_run iters=2 vs iters=1")
            assert (d1[n:] == POISON).all(), what + ": dev_run wrote past the last row"
            _first_diff(d1[:n], out, what + ": dev_run vs host")
            if op.status:
                assert (s1 == s2).all() and (s1[n:] == POISON).all(), what + ": statuses past n or between iters"
                _first_diff(s1[:n, None], st[:, None], what + ": dev_run vs host statuses")
            idx = samples[n]
            pos = np.searchsorted(rows, idx)
            _first_diff(out[idx], want_out[pos], what + ": host vs oracle")
            if op.status:
                _first_diff(st[idx, None], want_st[pos, None], what + ": host vs oracle statuses")
        # page-locked inputs and outputs at the size just past one full chunk (chunks of full size: no staging, and for the
        # variable-base DH ops twice the staged chunk)
        n = op.chunk + 1
        pins = []
        for x in ins:
            p = fq.pinned_empty((n, x.shape[1])); p[:] = x[:n]; pins.append(p)
        pout = fq.pinned_empty((n, op.out)); pout[:] = POISON
        pst = fq.pinned_empty((n,)) if op.status else None
        if pst is not None:
            pst[:] = POISON
        _host(op, pins, n, 1, fixed_base, out=pout, status=pst)
        _first_diff(np.asarray(pout), kept[0], name + ": pinned out= vs pageable")
        if op.status:
            _first_diff(np.asarray(pst)[:, None], kept[1][:, None], name + ": pinned status= vs pageable")
    finally:
        dev.free()


@pytest.mark.parametrize("name", sorted(OPS))
def test_host_path_on_all_gpus(fq, pool, fixed_base, name):
    """ndev = every visible GPU, pageable and page-locked (laid out for that many GPUs), against ndev = 1, one chunk past full."""
    nd = fq.device_count()
    if nd < 2:
        pytest.skip("one GPU: the ndev = all case needs two or more")
    op = OPS[name]
    n = op.chunk + 1
    ins = [x[:n] for x in _inputs(op, op.sizes()[-1], pool)]
    want = _host(op, ins, n, 1, fixed_base)
    got = _host(op, ins, n, nd, fixed_base)
    _first_diff(got[0], want[0], name + ": ndev=%d vs 1" % nd)
    pins = []
    for x in ins:
        p = fq.pinned_empty((n, x.shape[1]), ndev=nd); p[:] = x; pins.append(p)
    pout = fq.pinned_empty((n, op.out), ndev=nd)
    pst = fq.pinned_empty((n,), ndev=nd) if op.status else None
    _host(op, pins, n, nd, fixed_base, out=pout, status=pst)
    _first_diff(np.asarray(pout), want[0], name + ": pinned ndev=%d vs 1" % nd)
    if op.status:
        assert (got[1] == want[1]).all() and (np.asarray(pst) == want[1]).all()


@pytest.mark.parametrize("name", ["fp2_inv", "f25519_inv"])
def test_batched_inverse_refuses_out_aliasing_a(fq, name):
    """The batched inversions park prefix products in `out`, so fq_dev_run3 refuses out == a before any launch."""
    from fourq_b200 import device
    L = _lib()
    a = np.random.default_rng(3).integers(0, 256, (4096, 32), np.uint8)
    d = device.DeviceBuffer.from_host(0, a)
    ms = ctypes.c_float()
    assert L.lib().fq_dev_run3(L.DEVOP[name], 0, d.ptr, None, None, d.ptr, None, 4096, 1, ctypes.byref(ms)) == L.FQ_ERR_ARG
    assert b"alias" in L.lib().fq_last_error()
    assert (d.to_host((4096, 32)) == a).all()
    d.free()
