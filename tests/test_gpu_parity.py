"""GPU parity tests (run on the B200 with -m gpu).  Everything goes through the Python facade -> ctypes -> C ABI ->
CUDA kernels and is compared bit-for-bit with (a) the golden vectors generated from the reference's own code and
(b) the CPU oracle on seeded random inputs; at BASELINE sizes (2^20) size-independent properties are checked."""
import multiprocessing as mp
import os
import random

import numpy as np
import pytest

from oracle import fourq_oracle as O

pytestmark = pytest.mark.gpu
H = bytes.fromhex


@pytest.fixture(scope="module")
def fq():
    import fourq_b200
    assert fourq_b200.device_count() >= 1        # raises if the CUDA library or device is missing: no silent fallback
    return fourq_b200


def R(lst, width=None):
    return np.frombuffer(b"".join(lst), np.uint8).reshape(len(lst), -1).copy()


def hexrows(a):
    return [bytes(r).hex() for r in a]


# ---------------------------------------------------------------- golden vectors (from the reference's code)

@pytest.mark.parametrize("op", ["mul", "add", "sub"])
def test_fp2_binary_golden(fq, golden, op):
    rows = golden["fields"][op]
    got = getattr(fq.GFp2, op)(R([H(r[0]) for r in rows]), R([H(r[1]) for r in rows]))
    assert hexrows(got) == [r[2] for r in rows]


@pytest.mark.parametrize("op", ["sqr", "neg", "conj", "inv"])
def test_fp2_unary_golden(fq, golden, op):
    rows = golden["fields"][op]
    got = getattr(fq.GFp2, op)(R([H(r[0]) for r in rows]))
    assert hexrows(got) == [r[1] for r in rows]


@pytest.mark.parametrize("op", ["add", "sub", "mul", "sqr", "neg", "inv", "invsqrt"])
def test_fp_rows_golden_and_random(fq, golden, op):
    rows = golden["fp"][op]
    binary = len(rows[0]) == 3
    a = R([H(r[0]) for r in rows], 16)
    got = getattr(fq.GFp, op)(a, R([H(r[1]) for r in rows], 16)) if binary else getattr(fq.GFp, op)(a)
    assert hexrows(got) == [r[-1] for r in rows]
    rng = np.random.default_rng(11)
    n = 4096 if op in ("inv", "invsqrt") else 65536
    x = rng.integers(0, 256, (n, 16), np.uint8); y = rng.integers(0, 256, (n, 16), np.uint8)
    got = getattr(fq.GFp, op)(x, y) if binary else getattr(fq.GFp, op)(x)
    idx = range(0, n, 16)
    assert [bytes(got[j]) for j in idx] == [O.row_fp(op, bytes(x[j]), bytes(y[j]) if binary else None) for j in idx]


def test_codec_golden(fq, golden):
    c = golden["codec"]
    assert hexrows(fq.encode(R([H(r[0]) for r in c["encode"]]))) == [r[1] for r in c["encode"]]
    B = R([H(r[0]) for r in c["decode"]])
    keep = B.copy()
    XY, st = fq.decode(B)
    assert (B == keep).all()                     # no in-place mutation (the reference mutates, curve4q.py:56)
    assert [(int(s), x) for s, x in zip(st, hexrows(XY))] == [(r[1], r[2]) for r in c["decode"]]
    assert set(int(s) for s in st) == {0, 1, 2, 3, 4}


@pytest.mark.parametrize("alg", ["windowed", "endo"])
def test_scalar_mult_golden(fq, golden, alg):
    """MUL_windowed / MUL_endo based entry points: the reference asserts both give the same points (curve4q.py:706-762)."""
    m = golden["mul"]
    assert hexrows(fq.MUL_base(R([H(r[0]) for r in m["mul_base"]]), algorithm=alg)) == [r[1] for r in m["mul_base"]]
    out, st = fq.DH_base(R([H(r[0]) for r in m["dh_base"]]), algorithm=alg)
    assert [(int(s), o) for s, o in zip(st, hexrows(out))] == [(r[1], r[2]) for r in m["dh_base"]]
    out, st = fq.DH(R([H(r[0]) for r in m["dh"]]), R([H(r[1]) for r in m["dh"]]), algorithm=alg)
    assert [(int(s), o) for s, o in zip(st, hexrows(out))] == [(r[2], r[3]) for r in m["dh"]]
    assert set(int(s) for s in st) == {0, 1, 2, 3, 4, 5}
    dh_aff = fq.DH_windowed if alg == "windowed" else fq.DH_endo
    out, st = dh_aff(R([H(r[0]) for r in m["dh_affine"]]), R([H(r[1]) for r in m["dh_affine"]]))
    assert [(int(s), o) for s, o in zip(st, hexrows(out))] == [(r[2], r[3]) for r in m["dh_affine"]]


def test_strict_select_mode_gives_identical_outputs(fq):
    """fq_set_select_mode: the strict scan (default: every lane loads every table entry, SEL per word) and the masked loads
    (opt-in, predicated LDS); every scalar-multiplication kernel must give the same bytes in both modes."""
    rng = np.random.default_rng(61)
    n = 20000
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
    pub[::11] = rng.integers(0, 256, (len(pub[::11]), 32), np.uint8)
    default = fq.get_select_mode()
    if os.environ.get("FQ_STRICT_SELECT") is None:
        assert default is True                       # the library default is the strict scan (no digit-dependent memory activity)
    ref = {}
    try:
        for strict in (True, False):
            fq.set_select_mode(strict)
            assert fq.get_select_mode() is strict
            got = {"dh_endo": fq.DH(k, pub, algorithm="endo"), "dh_win": fq.DH(k, pub, algorithm="windowed")}
            for alg in ("comb", "endo", "windowed"):
                got["mul_" + alg] = (fq.MUL_base(k, algorithm=alg),)
                got["dhb_" + alg] = fq.DH_base(k, algorithm=alg)
            if strict:
                ref = got
            else:
                for name in ref:
                    assert all((a == b).all() for a, b in zip(ref[name], got[name])), name
    finally:
        fq.set_select_mode(default)
    from oracle import c_oracle as C
    want, wst = C.dh(k, pub)
    assert (ref["dh_endo"][0] == want).all() and (ref["dh_endo"][1] == wst).all()


def test_point_on_curve(fq, golden):
    from oracle import c_oracle as C
    import fourq_b200.curve4q as c4
    rng = np.random.default_rng(81)
    pub = fq.MUL_base(rng.integers(0, 256, (5000, 32), np.uint8))
    xy, st = fq.decode(pub)
    assert not st.any() and c4.PointOnCurve(xy).all()
    mixed = xy.copy(); mixed[::3, rng.integers(0, 64)] ^= 0x10
    mixed = np.concatenate([mixed, rng.integers(0, 256, (999, 64), np.uint8), np.zeros((1, 64), np.uint8)])    # non-canonical halves too
    got = c4.PointOnCurve(mixed)
    assert (got == C.on_curve(mixed)).all() and got.any() and not got.all()


def test_decode_spec_opt_in(fq, golden):
    rows = golden["codec"]["decode"]
    low = [O.encode(x, y) for x, y in (((0, 0), (1, 0)), ((0, 0), (O.P127 - 1, 0)), ((0, 1), (0, 0)), ((0, O.P127 - 1), (0, 0)))]
    enc = R([H(r[0]) for r in rows] + low)
    xy, st = fq.decode(enc, spec=True)
    want = [O.row_decode(bytes(e), spec=True) for e in enc]
    assert [(bytes(a), int(b)) for a, b in zip(xy, st)] == want
    assert not st[-4:].any() and 3 not in set(int(s) for s in st)
    xy0, st0 = fq.decode(enc)                                      # default stays bit-compatible: the four are status 3
    assert list(st0[-4:]) == [3, 3, 3, 3]
    keep = st0 != 3
    assert (xy[keep] == xy0[keep]).all() and (st[keep] == st0[keep]).all()


def test_baseline_config1_reference_vectors(fq, golden):
    """BASELINE.json configs[0]: 1,024 random scalars x the base point, outputs of the reference's own DH_windowed
    (tests/golden/cfg1.json), through every fixed-base algorithm and through the variable-base kernels on encode(G)."""
    k = np.random.default_rng(1).integers(0, 256, (1024, 32), np.uint8)
    want = golden["cfg1"]["out"]
    for alg in ("comb", "windowed", "endo"):
        out, st = fq.DH_base(k, algorithm=alg)
        assert not st.any() and hexrows(out) == want, alg
    Genc = np.tile(np.frombuffer(O.encode(O.GX, O.GY), np.uint8), (1024, 1))
    for alg in ("endo", "windowed"):
        out, st = fq.DH(k, Genc, algorithm=alg)
        assert not st.any() and hexrows(out) == want, alg


def test_fixed_base_comb_golden(fq, golden):
    """Per-digit tables (SURVEY 8f-2): same bytes as MUL_*(m, G, table) / DH_*(m, G, table=T392), incl. edge scalars."""
    m = golden["mul"]
    assert hexrows(fq.MUL_base(R([H(r[0]) for r in m["mul_base"]]), algorithm="comb")) == [r[1] for r in m["mul_base"]]
    out, st = fq.DH_base(R([H(r[0]) for r in m["dh_base"]]), algorithm="comb")
    assert [(int(s), o) for s, o in zip(st, hexrows(out))] == [(r[1], r[2]) for r in m["dh_base"]]
    assert 5 in set(int(s) for s in st)                       # scalars = 0 mod N are rejected as in curve4q.py:459


def test_reference_mulP_chain(fq, golden):
    """curve4q.py:549-567: 1000 chained MUL_windowed from G end at mulP, i.e. [prod c_i mod N]G == mulP."""
    m = golden["mul"]
    prod = 1
    for k in m["mulP_chain_scalars"]:
        prod = prod * int.from_bytes(H(k), "little") % O.N
    P = O.xy_from_bytes(H(m["mulP_affine"]))
    for alg in ("windowed", "endo", "comb"):
        got = fq.MUL_base(fq.curve4q.pack_scalars([prod]), algorithm=alg)
        assert bytes(got[0]) == O.encode(P[0], P[1])
    # [2^1000]G and the addition KAT (curve4q.py:516-547), via scalars
    for name, k in (("doubleP_affine", pow(2, 1000, O.N)), ("P1000_affine", 1002)):
        P = O.xy_from_bytes(H(m[name]))
        assert bytes(fq.MUL_base(fq.curve4q.pack_scalars([k]))[0]) == O.encode(P[0], P[1])


def test_strict_mode_raises_reference_messages(fq, golden):
    c = golden["codec"]
    bad = [r for r in c["decode"] if r[1] == 4][0]
    with pytest.raises(Exception, match="Point not on curve"):
        fq.decode(R([H(bad[0])]), strict=True)
    quirk = [r for r in c["decode"] if r[1] == 3][0]
    with pytest.raises(AttributeError):
        fq.decode(R([H(quirk[0])]), strict=True)
    with pytest.raises(Exception, match="neutral point"):
        fq.DH_base(fq.curve4q.pack_scalars([O.N]), strict=True)


def test_x25519_golden_and_rfc(fq, golden, x25519_kat):
    rows = golden["x25519"]["x25519"]
    got = fq.x25519(R([H(r[0]) for r in rows]), R([H(r[1]) for r in rows]))
    assert hexrows(got) == [r[2] for r in rows]
    kat = x25519_kat                              # the reference's own known answers: curve25519.py:96-107 (rfc-0/1), :131-149 (test_dh)
    assert hexrows(fq.x25519(R([H(r[0]) for r in kat]), R([H(r[1]) for r in kat]))) == [r[2] for r in kat]
    k = u = R([bytes([9] + [0] * 31)])
    for i in range(1000):                        # RFC 7748 5.2, curve25519.py:104-124
        k, u = fq.x25519(k, u), k
        if i == 0:
            assert bytes(k[0]).hex() == "422c8e7a6227d7bca1350b3e2bb7279f7897b87bb6854b783c60e80311ae3079"
    assert bytes(k[0]).hex() == "684cf59ba83309552800ef566f2f4d3c1c3887c49360e3875f2eb94d99532c51"


def _oracle_x25519(args):
    return O.x25519(args[0], args[1])


def test_x25519_random_and_special_vs_oracle(fq):
    """Config 5's X25519 kernel on 2,048 random (k, u) rows and on special u coordinates (0, 1, p-1, p, p+1, 2^255-1, the
    low-order points of RFC 7748 section 6 notes, all-ones limbs) x special scalars, against the Python oracle."""
    rng = np.random.default_rng(91)
    p = (1 << 255) - 19
    us = [0, 1, 2, 9, p - 1, p, p + 1, (1 << 255) - 1, (1 << 256) - 1, 1 << 255, (1 << 254) + 7,
          325606250916557431795983626356110631294008115727848805560023387167927233504,          # order 8
          39382357235489614581723060781553021112529911719440698176882885853963445705823,        # order 8
          int("ffffffff00000000" * 4, 16), int("00000000ffffffff" * 4, 16)]
    ks = [0, 1, 8, (1 << 254), (1 << 255) - 1, (1 << 256) - 1, int("a5" * 32, 16), int("0f" * 32, 16)]
    kk = [int(a).to_bytes(32, "little") for a in ks for _ in us] + [bytes(r) for r in rng.integers(0, 256, (2048, 32), np.uint8)]
    uu = [int(b).to_bytes(32, "little") for _ in ks for b in us] + [bytes(r) for r in rng.integers(0, 256, (2048, 32), np.uint8)]
    got = fq.x25519(R(kk), R(uu))
    with _pool() as pool:
        want = pool.map(_oracle_x25519, list(zip(kk, uu)), chunksize=32)
    assert [bytes(r) for r in got] == want


# ---------------------------------------------------------------- seeded random vs the oracle

def _oracle_fp2(args):
    op, a, b = args
    return O.row_fp2(op, a, b)


def _oracle_dh(args):
    return O.row_dh(*args)


def _oracle_mul_base(k):
    return O.row_mul_base(k)


def _pool():
    return mp.get_context("fork").Pool(min(16, os.cpu_count() or 1))


def test_fp2_random_65536_vs_oracle(fq):
    rng = np.random.default_rng(2)
    n = 1 << 16
    a = rng.integers(0, 256, (n, 32), np.uint8); b = rng.integers(0, 256, (n, 32), np.uint8)
    edge = [0, 1, O.P127 - 1, O.P127, O.P127 + 1, 1 << 127, (1 << 128) - 1, (1 << 64) - 1, (1 << 64) + 1]
    i = 0
    for x in edge:
        for y in edge:
            a[i] = np.frombuffer(x.to_bytes(16, "little") + y.to_bytes(16, "little"), np.uint8)
            b[i] = np.frombuffer(y.to_bytes(16, "little") + x.to_bytes(16, "little"), np.uint8)
            i += 1
    with _pool() as pool:
        for op in ("mul", "sqr", "add", "sub"):
            got = getattr(fq.GFp2, op)(a, b) if op in ("mul", "add", "sub") else fq.GFp2.sqr(a)
            want = pool.map(_oracle_fp2, [(op, bytes(a[j]), bytes(b[j])) for j in range(n)], chunksize=2048)
            assert [bytes(r) for r in got] == want, op
        got = fq.GFp2.inv(a[:4096])
        want = pool.map(_oracle_fp2, [("inv", bytes(a[j]), None) for j in range(4096)], chunksize=256)
        assert [bytes(r) for r in got] == want


def test_dh_random_4096_vs_oracle(fq):
    rng = np.random.default_rng(3)
    n = 4096
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(np.random.default_rng(4).integers(0, 256, (n, 32), np.uint8))
    pub[::7] = rng.integers(0, 256, (len(pub[::7]), 32), np.uint8)      # arbitrary strings: ~half fail to decode
    out, st = fq.DH(k, pub, algorithm="windowed")
    out2, st2 = fq.DH(k, pub, algorithm="endo")
    with _pool() as pool:
        want = pool.map(_oracle_dh, [(bytes(k[j]), bytes(pub[j])) for j in range(n)], chunksize=32)
        assert [(bytes(o), int(s)) for o, s in zip(out, st)] == want
        assert [(bytes(o), int(s)) for o, s in zip(out2, st2)] == want
        kb = rng.integers(0, 256, (1024, 32), np.uint8)
        assert [bytes(r) for r in fq.MUL_base(kb)] == pool.map(_oracle_mul_base, [bytes(r) for r in kb], chunksize=16)


# ---------------------------------------------------------------- BASELINE sizes: properties that need no oracle

def test_full_size_properties_2_20(fq):
    n = 1 << 20
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, (n, 32), np.uint8); b = rng.integers(0, 256, (n, 32), np.uint8)
    A, sa = fq.DH_base(a, algorithm="windowed"); Bp, sb = fq.DH_base(b, algorithm="endo")       # [392a]G, [392b]G
    assert not sa.any() and not sb.any()
    AB, s1 = fq.DH(a, Bp, algorithm="windowed"); BA, s2 = fq.DH(b, A, algorithm="endo")           # DH symmetry (curve4q.py:725-738)
    assert not s1.any() and not s2.any()
    assert (AB == BA).all()
    AB2, _ = fq.DH(a, Bp, algorithm="endo")                              # windowed == endo on 2^20 rows (curve4q.py:706-762)
    assert (AB2 == AB).all()
    assert (fq.MUL_base(a, algorithm="windowed") == fq.MUL_base(a, algorithm="endo")).all()
    assert (fq.MUL_base(a, algorithm="comb") == fq.MUL_base(a, algorithm="endo")).all()     # per-digit tables, 2^20 rows
    Ac, sc = fq.DH_base(a, algorithm="comb")
    assert not sc.any() and (Ac == A).all()
    # fixed base == variable base on G (curve4q.py:743-762)
    Genc = np.tile(np.frombuffer(O.encode(O.GX, O.GY), np.uint8), (n, 1))
    viaG, s3 = fq.DH(a, Genc)
    assert not s3.any() and (viaG == A).all()
    # encode(decode(x)) round trip on 2^20 valid points, and every row of the batch is distinct work
    XY, s4 = fq.decode(A)
    assert not s4.any() and (fq.encode(XY) == A).all()
    # field identities at size: (a*b)*inv(b) == a for invertible b; a^2 == a*a
    fa = a.copy(); fb = b.copy(); fa[:, 15] &= 0x7F; fa[:, 31] &= 0x7F; fb[:, 15] &= 0x7F; fb[:, 31] &= 0x7F
    prod = fq.GFp2.mul(fa, fb)
    assert (fq.GFp2.sqr(fa) == fq.GFp2.mul(fa, fa)).all()
    assert (fq.GFp2.mul(prod, fq.GFp2.inv(fb)) == fq.GFp2.mul(fa, fq.GFp2.mul(fb, fq.GFp2.inv(fb)))).all()


def test_full_size_bit_exact_vs_c_oracle(fq):
    """Every row of a BASELINE-size batch against oracle/fourq_oracle.c (pinned to the reference's golden vectors by
    tests/test_oracle_c.py): 2^20 variable-base DH rows incl. undecodable strings, 2^20 fixed-base rows."""
    from oracle import c_oracle as C
    n = 1 << 20
    rng = np.random.default_rng(41)
    k = rng.integers(0, 256, (n, 32), np.uint8)
    kp = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(kp)                                            # comb kernel
    assert (pub == C.mul_base(kp)).all()
    pub[::97] = rng.integers(0, 256, (len(pub[::97]), 32), np.uint8)   # ~1 % arbitrary strings: every decode failure class
    want, wst = C.dh(k, pub)
    got, st = fq.DH(k, pub)                                          # endo
    assert (st == wst).all() and (got == want).all()
    assert set(np.unique(wst)) >= {0, 4}
    m = 1 << 18
    got, st = fq.DH(k[:m], pub[:m], algorithm="windowed")
    assert (st == wst[:m]).all() and (got == want[:m]).all()
    gb, sb = fq.DH_base(k[:m])
    wb, wsb = C.dh_base(k[:m])
    assert (sb == wsb).all() and (gb == wb).all()


def test_adversarial_grid_vs_c_oracle(fq):
    """tests/adversarial.py: limb patterns built to break carry chains, folds, recoding and decoding -- GF(p^2) and GF(p) ops on
    boundary and non-canonical values, and ~1,000 DH rows of special scalars x valid / invalid points, in both algorithms and
    both table-selection modes, against the C oracle."""
    import adversarial as A
    from oracle import c_oracle as C
    a, b = A.fp2_grid()
    for op in ("mul", "add", "sub"):
        assert (getattr(fq.GFp2, op)(a, b) == C.fp2(op, a, b)).all(), op
        assert (getattr(fq.GFp, op)(a[:, :16], b[:, :16]) == C.fp(op, a[:, :16], b[:, :16])).all(), op
    for op in ("sqr", "inv", "neg", "conj"):
        ar = a.copy() if op in ("sqr", "inv") else C.fp2("add", a, np.zeros_like(a))      # neg / conj: reduced input as in the reference
        assert (getattr(fq.GFp2, op)(ar) == C.fp2(op, ar)).all(), op
    for op in ("sqr", "inv", "invsqrt"):
        assert (getattr(fq.GFp, op)(a[:, :16]) == C.fp(op, a[:, :16])).all(), op
    k, enc = A.grid()
    want, wst = C.dh(k, enc)
    assert set(int(x) for x in wst) >= {0, 3, 4, 5}
    default = fq.get_select_mode()
    try:
        for strict in (False, True):
            fq.set_select_mode(strict)
            for alg in ("endo", "windowed"):
                out, st = fq.DH(k, enc, algorithm=alg)
                assert (st == wst).all() and (out == want).all(), (strict, alg)
    finally:
        fq.set_select_mode(default)
    ks = k[:: 7]
    for alg in ("comb", "endo", "windowed"):
        assert (fq.MUL_base(ks, algorithm=alg) == C.mul_base(ks)).all(), alg
        gb, sb = fq.DH_base(ks, algorithm=alg); wb, wsb = C.dh_base(ks)
        assert (gb == wb).all() and (sb == wsb).all(), alg


def test_ragged_and_empty_batches(fq):
    rng = np.random.default_rng(6)
    assert fq.MUL_base(np.zeros((0, 32), np.uint8)).shape == (0, 32)
    out, st = fq.DH(np.zeros((0, 32), np.uint8), np.zeros((0, 32), np.uint8))
    assert out.shape == (0, 32) and st.shape == (0,)
    k = rng.integers(0, 256, ((1 << 17) + 131, 32), np.uint8)            # crosses chunk boundaries of the ramped schedule, not a multiple of 128
    full = fq.MUL_base(k)
    for n in (1, 31, 127, 129, 1000):
        assert (fq.MUL_base(k[:n]) == full[:n]).all()
    assert (fq.MUL_base(k[-200:]) == full[-200:]).all()
    # non-contiguous input is accepted (copied)
    assert (fq.MUL_base(k[::2][:64]) == full[::2][:64]).all()


def _oracle_dh_affine(args):
    return O.row_dh_affine(args[0], args[1], mul=O.mul_endo if args[2] == "endo" else O.mul_windowed)


def test_dh_ragged_batches_and_failures_next_to_good_rows(fq):
    """Variable-base DH on batches that are not multiples of 128 or 4, with every failure class in the same inversion
    groups as good rows (k_dh_finish shares one inversion between 4 rows): decode failures, the reference's t == 0 quirk,
    neutral results (k = 0 mod N), against the oracle row by row; also the affine entry points and y_only."""
    rng = np.random.default_rng(21)
    n = 1003
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
    pub[::5] = rng.integers(0, 256, (len(pub[::5]), 32), np.uint8)                      # arbitrary strings
    quirk = np.frombuffer(O.encode((0, 0), (1, 0)), np.uint8)                          # (0, 1): status 3 in the reference
    pub[3::50] = quirk
    for j, m in zip(range(7, n, 40), [0, O.N, 2 * O.N, 5 * O.N, O.N - 1, O.N + 1, 1, 2] * 4):
        k[j] = np.frombuffer(int(m).to_bytes(32, "little"), np.uint8)
        pub[j] = np.frombuffer(O.encode(O.GX, O.GY), np.uint8)
    with _pool() as pool:
        want = pool.map(_oracle_dh, [(bytes(k[j]), bytes(pub[j])) for j in range(n)], chunksize=16)
        assert {s for _, s in want} >= {0, 3, 4, 5}
        for alg in ("endo", "windowed"):
            for m in (n, 1, 3, 5, 127, 129, 515):
                out, st = fq.DH(k[:m], pub[:m], algorithm=alg)
                assert [(bytes(o), int(s)) for o, s in zip(out, st)] == want[:m], (alg, m)
        ysec, st = fq.DH(k, pub, y_only=True)
        assert [bytes(r) for r in ysec] == [bytes(o[:31] + bytes([o[31] & 0x7F])) for o, _ in want]
        # affine entry points: valid points from decode, plus points off the curve (status 4)
        XY, sd = fq.decode(pub)
        XY[11::13, 5] ^= 1
        want_aff = pool.map(_oracle_dh_affine, [(bytes(k[j]), bytes(XY[j]), "endo") for j in range(0, n, 3)], chunksize=16)
        for fn in (fq.DH_endo, fq.DH_windowed):
            out, st = fn(k, XY)
            assert [(bytes(out[j]), int(st[j])) for j in range(0, n, 3)] == want_aff, fn.__name__


def test_device_resident_batch_larger_than_one_launch_group(fq):
    """fq_dev_run on more rows than one launch group of the DH kernels (2^22): the batches must tile the buffers exactly."""
    from fourq_b200 import device as fqdev
    n = (1 << 22) + 777
    rng = np.random.default_rng(22)
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
    dk = fqdev.DeviceBuffer.from_host(0, k); dp = fqdev.DeviceBuffer.from_host(0, pub)
    do = fqdev.DeviceBuffer(0, n * 32); ds = fqdev.DeviceBuffer(0, n)
    fqdev.dev_run("dh_endo", 0, dk, dp, do, ds, n)
    got, st = do.to_host((n, 32)), ds.to_host((n,))
    want, wst = fq.DH(k, pub)                                   # host path: ramped chunks of up to 454,656 rows
    assert not st.any() and not wst.any() and (got == want).all()
    dko = fqdev.DeviceBuffer(0, n * 32)
    fqdev.dev_run("mul_base_comb", 0, dk, None, dko, None, n)
    assert (dko.to_host((n, 32)) == fq.MUL_base(k)).all()


def test_argument_errors_are_reported_not_swallowed(fq):
    rng = np.random.default_rng(71)
    k = rng.integers(0, 256, (8, 32), np.uint8)
    with pytest.raises(fq.FourQError, match="ndev"):
        fq.MUL_base(k, ndev=fq.device_count() + 1)
    with pytest.raises(ValueError):
        fq.DH(k, k[:4])
    with pytest.raises(ValueError):
        fq.DH(k, np.zeros((8, 31), np.uint8))
    with pytest.raises(TypeError):
        fq.MUL_base(k.astype(np.int32))
    with pytest.raises(ValueError):
        fq.MUL_base(k, algorithm="nope")
    with pytest.raises(ValueError):
        fq.MUL_base(k, out=np.zeros((7, 32), np.uint8))
    from fourq_b200 import _lib
    assert _lib.lib().fq_fp_op(99, _lib.ptr(k), None, _lib.ptr(k), 1, 1) == _lib.FQ_ERR_ARG
    assert _lib.lib().fq_set_select_mode(7) == _lib.FQ_ERR_ARG
    assert b"select mode" in _lib.lib().fq_last_error()
    assert _lib.lib().fq_dh(None, None, None, None, 5, 1) == _lib.FQ_ERR_ARG          # null buffers with n > 0
    assert _lib.lib().fq_dh(None, None, None, None, 0, 1) == _lib.FQ_OK               # n = 0 touches nothing


def test_concurrent_callers_and_trim(fq):
    """Two Python threads call different entry points at the same time (the engine serialises them); fq_trim releases the
    buffers and the next call works again with the same results."""
    import threading
    rng = np.random.default_rng(95)
    k = rng.integers(0, 256, (30000, 32), np.uint8)
    pub = fq.MUL_base(k)
    want_dh = fq.DH(k, pub)
    want_mul = fq.MUL_base(k, algorithm="endo")
    want_x = fq.x25519(k, pub)
    res = {}

    def worker(name, fn):
        for _ in range(4):
            res[name] = fn()
    ts = [threading.Thread(target=worker, args=("dh", lambda: fq.DH(k, pub))),
          threading.Thread(target=worker, args=("mul", lambda: fq.MUL_base(k, algorithm="endo"))),
          threading.Thread(target=worker, args=("x", lambda: fq.x25519(k, pub)))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert (res["dh"][0] == want_dh[0]).all() and (res["dh"][1] == want_dh[1]).all() and (res["mul"] == want_mul).all()
    assert (res["x"] == want_x).all()
    fq.trim()
    again = fq.DH(k, pub)
    assert (again[0] == want_dh[0]).all() and (fq.MUL_base(k) == pub).all()


def test_pinned_host_buffers(fq):
    rng = np.random.default_rng(8)
    k = fq.pinned_empty((5000, 32)); k[:] = rng.integers(0, 256, (5000, 32), np.uint8)
    assert (fq.MUL_base(k) == fq.MUL_base(np.array(k))).all()


def test_multi_gpu_slices_match_single(fq):
    if fq.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    rng = np.random.default_rng(9)
    k = rng.integers(0, 256, (100001, 32), np.uint8)
    pub = fq.MUL_base(k, ndev=1)
    assert (fq.MUL_base(k, ndev=2) == pub).all()
    pub[::101] = rng.integers(0, 256, (len(pub[::101]), 32), np.uint8)
    k2 = rng.integers(0, 256, (100001, 32), np.uint8)
    o1, s1 = fq.DH(k2, pub, ndev=1)
    for g in range(2, min(fq.device_count(), 8) + 1):
        og, sg = fq.DH(k2, pub, ndev=g)                      # contiguous slices of ceil(n/g) rows, ragged last slice
        assert (og == o1).all() and (sg == s1).all(), g


# ---------------------------------------------------------------- round 2 additions

def test_select_and_fp2_invsqrt_golden_and_random(fq, golden):
    """fq_fp_select / fq_fp2_select / fq_fp2_invsqrt (fields.py:59-64, :236-238, :201-230) against vectors produced by the reference
    and against the oracle on random rows."""
    g = golden["select"]
    for key, cls in (("fp_select", fq.GFp), ("fp2_select", fq.GFp2)):
        rows = g[key]
        got = cls.select(np.array([r[0] for r in rows], np.uint8), R([H(r[1]) for r in rows]), R([H(r[2]) for r in rows]))
        assert hexrows(got) == [r[3] for r in rows]
    rows = g["fp2_invsqrt"]
    assert hexrows(fq.GFp2.invsqrt(R([H(r[0]) for r in rows]))) == [r[1] for r in rows]
    rng = np.random.default_rng(77)
    n = 100003
    x = rng.integers(0, 256, (n, 32), np.uint8); y = rng.integers(0, 256, (n, 32), np.uint8)
    c = rng.integers(0, 2, n, np.uint8)
    assert (fq.GFp2.select(c, x, y) == np.where(c.reshape(-1, 1) == 1, x, y)).all()
    x16, y16 = np.ascontiguousarray(x[:, :16]), np.ascontiguousarray(y[:, 16:])
    assert (fq.GFp.select(c, x16, y16) == np.where(c.reshape(-1, 1) == 1, x16, y16)).all()
    a = rng.integers(0, 256, (4096, 32), np.uint8)
    a[::7, 16:] = 0                                                  # the GF(p) branch
    got = fq.GFp2.invsqrt(a)
    assert [bytes(r) for r in got] == [O.row_fp2("invsqrt", bytes(r)) for r in a]
    # where the input is a square the result really is an inverse square root: a * r^2 == 1
    chk = fq.GFp2.mul(a, fq.GFp2.sqr(got))
    one = np.zeros(32, np.uint8); one[0] = 1
    assert (chk == one).all(axis=1).sum() > 1000


def test_fp2_inv_shared_inversion_with_zero_rows(fq):
    """k_fp2_inv_batched: one chain per 16 rows; zeros (in every disguise) inside the groups, ragged sizes."""
    rng = np.random.default_rng(78)
    p = O.P127
    for n in (1, 15, 16, 17, 1023, 70001):
        a = rng.integers(0, 256, (n, 32), np.uint8)
        z = rng.random(n) < 0.1
        a[z] = 0
        a[rng.random(n) < 0.03] = np.frombuffer(p.to_bytes(16, "little") * 2, np.uint8)          # (p, p) = zero
        got = fq.GFp2.inv(a)
        idx = list(range(0, n, max(1, n // 300)))
        assert [bytes(got[i]) for i in idx] == [O.row_fp2("inv", bytes(a[i])) for i in idx]
        assert (got[(a == 0).all(axis=1)] == 0).all()


def test_gfp25519_field_ops_golden_random_and_identities(fq, golden):
    """fq_fp25519_op (fields.py:267-362 GFp25519.add/sub/mul/sqr/inv, compare.py:14-49's other column): the reference's vectors,
    random unreduced rows against the oracle, zeros in every disguise through the shared inversion, and x * inv(x) == 1 at size."""
    g = golden["f25519"]
    for op in ("add", "sub", "mul"):
        rows = g[op]
        assert hexrows(getattr(fq.GFp25519, op)(R([H(r[0]) for r in rows]), R([H(r[1]) for r in rows]))) == [r[2] for r in rows], op
    for op in ("sqr", "inv"):
        rows = g[op]
        assert hexrows(getattr(fq.GFp25519, op)(R([H(r[0]) for r in rows]))) == [r[1] for r in rows], op
    rng = np.random.default_rng(2519)
    q = O.P25519
    for n in (1, 17, 4099):
        a = rng.integers(0, 256, (n, 32), np.uint8); b = rng.integers(0, 256, (n, 32), np.uint8)
        a[rng.random(n) < 0.1] = 0
        a[rng.random(n) < 0.05] = np.frombuffer(q.to_bytes(32, "little"), np.uint8)
        a[rng.random(n) < 0.05] = np.frombuffer((2 * q).to_bytes(32, "little"), np.uint8)
        for op in ("add", "sub", "mul"):
            assert [bytes(r) for r in getattr(fq.GFp25519, op)(a, b)] == [O.row_f25519(op, bytes(x), bytes(y)) for x, y in zip(a, b)], op
        for op in ("sqr", "inv"):
            assert [bytes(r) for r in getattr(fq.GFp25519, op)(a)] == [O.row_f25519(op, bytes(x)) for x in a], op
    n = (1 << 20) + 5
    a = rng.integers(0, 256, (n, 32), np.uint8)
    one = np.zeros(32, np.uint8); one[0] = 1
    assert (fq.GFp25519.mul(a, fq.GFp25519.inv(a)) == one).all()
    assert (fq.GFp25519.sub(fq.GFp25519.add(a, a[::-1].copy()), a[::-1].copy()) == fq.GFp25519.add(a, np.zeros_like(a))).all()
    assert (fq.GFp25519.sqr(a) == fq.GFp25519.mul(a, a)).all()
    with pytest.raises(fq.FourQError):
        from fourq_b200 import _lib
        _lib.check(_lib.lib().fq_fp25519_op(6, _lib.ptr(a), None, _lib.ptr(a), 4, 1))


def test_pageable_and_pinned_paths_agree_over_many_chunks(fq):
    """The host engine's staging of pageable inputs/outputs (capi.cu feeder / drainer) against page-locked buffers, on a batch that
    spans several ramped chunks; also rejects a device pointer as a host buffer."""
    rng = np.random.default_rng(79)
    n = 1_300_007
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pk = fq.pinned_empty((n, 32)); pk[:] = k
    po = fq.pinned_empty((n, 32))
    a = fq.MUL_base(k)                      # pageable in, pageable out
    fq.MUL_base(pk, out=po)                 # pinned in, pinned out
    b = fq.MUL_base(pk)                     # pinned in, pageable out
    assert (a == po).all() and (a == b).all()
    from oracle import c_oracle as C
    want, _ = C.dh(k[:2048], a[:2048])
    got, st = fq.DH(k[:2048], a[:2048])
    assert (got == want).all() and not st.any()
    from fourq_b200 import _lib, device
    d = device.DeviceBuffer(0, 64)
    assert _lib.lib().fq_fp2_sqr(_lib.ptr(k), d.ptr, 2, 1) == _lib.FQ_ERR_ARG
    assert b"device memory" in _lib.lib().fq_last_error()


def test_on_curve_device_op_is_bound(fq):
    from fourq_b200 import _lib, device
    assert _lib.DEVOP["on_curve"] == 30
    xy = R([O.xy_to_bytes(((O.GX), (O.GY))), bytes(64)])
    d_in = device.DeviceBuffer.from_host(0, xy); d_out = device.DeviceBuffer(0, 2)
    device.dev_run("on_curve", 0, d_in, None, d_out, None, 2)
    assert list(d_out.to_host((2,))) == [1, 0]


def test_sliced_pinned_arrays_and_rows_per_device(fq):
    """pinned_empty(..., ndev=N) (fq_host_alloc_sliced: NUMA placement where the platform allows, always page-locked) and the report of
    who processed what (fq_last_rows_per_device); with several GPUs the slices may be uneven (speed-proportional, work stealing) but
    the bytes never change."""
    from fourq_b200 import device
    g = min(fq.device_count(), 8)
    rng = np.random.default_rng(80)
    n = 600_011
    k = fq.pinned_empty((n, 32), ndev=max(g, 2)); k[:] = rng.integers(0, 256, (n, 32), np.uint8)
    out = fq.pinned_empty((n, 32), ndev=max(g, 2))
    ref = fq.MUL_base(np.array(k))
    for ndev in sorted({1, g}):
        for _ in range(3):                                   # later calls use the speeds measured by the earlier ones
            out[:] = 0
            fq.MUL_base(k, out=out, ndev=ndev)
            assert (out == ref).all()
            rows = device.last_rows_per_device(ndev)
            assert sum(rows) == n and all(r > 0 for r in rows), rows
