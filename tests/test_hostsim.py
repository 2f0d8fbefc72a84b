"""CPU checks of the DEVICE algorithms (fourq_b200/csrc/*.cuh) through tests/hostsim: the same headers compiled with
-DFQ_HOSTSIM, every PTX primitive emulated with its carry flag.  Compared with the golden vectors generated from the
reference and with the oracle on seeded random and edge inputs.  Test infrastructure only (the product has no CPU path)."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import fourq_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
H = bytes.fromhex
OPS = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4, "neg": 5, "conj": 6}


@pytest.fixture(scope="module")
def sim():
    so = os.path.join(HERE, "hostsim", "libfq_hostsim.so")
    srcs = [os.path.join(HERE, "hostsim", "hostsim.cpp")] + [
        os.path.join(HERE, "..", "fourq_b200", "csrc", f) for f in os.listdir(os.path.join(HERE, "..", "fourq_b200", "csrc")) if f.endswith(".cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(s) for s in srcs):
        subprocess.check_call([os.path.join(HERE, "hostsim", "build.sh")])
    return ctypes.CDLL(so)


def _rows(lst):
    return np.frombuffer(b"".join(lst), dtype=np.uint8).copy()


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def fp2_op(sim, op, A, B=None):
    a = _rows(A); out = np.zeros_like(a)
    b = _rows(B) if B is not None else None
    assert sim.sim_fp2_op(OPS[op], _p(a), _p(b) if b is not None else None, _p(out), ctypes.c_size_t(len(A))) == 0
    return [bytes(out[32 * i:32 * i + 32]) for i in range(len(A))]


@pytest.mark.parametrize("op", ["mul", "add", "sub"])
def test_fp2_binary_golden(sim, golden, op):
    rows = golden["fields"][op]
    got = fp2_op(sim, op, [H(r[0]) for r in rows], [H(r[1]) for r in rows])
    assert [g.hex() for g in got] == [r[2] for r in rows]


@pytest.mark.parametrize("op", ["sqr", "neg", "conj", "inv"])
def test_fp2_unary_golden(sim, golden, op):
    rows = golden["fields"][op]
    got = fp2_op(sim, op, [H(r[0]) for r in rows])
    assert [g.hex() for g in got] == [r[1] for r in rows]


FPOPS = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4, "neg": 5, "invsqrt": 6}


@pytest.mark.parametrize("op", ["add", "sub", "mul", "sqr", "neg", "inv", "invsqrt"])
def test_fp_rows_golden(sim, golden, op):
    rows = golden["fp"][op]
    a = _rows([H(r[0]) for r in rows]); out = np.zeros_like(a)
    b = _rows([H(r[1]) for r in rows]) if len(rows[0]) == 3 else None
    assert sim.sim_fp_row_op(FPOPS[op], _p(a), _p(b) if b is not None else None, _p(out), ctypes.c_size_t(len(rows))) == 0
    assert [bytes(out[16 * i:16 * i + 16]).hex() for i in range(len(rows))] == [r[-1] for r in rows]


def test_fp2_random_and_adversarial_vs_oracle(sim):
    rng = random.Random(7)
    p = O.P127
    special = [0, 1, 2, p - 1, p, p - 2, 1 << 126, (1 << 126) - 1, (1 << 64) - 1, (1 << 64) + 1, (1 << 96) - 1, 0xFFFFFFFF,
               (1 << 127) - (1 << 32), (1 << 127) - (1 << 64) - 1, 0xFFFFFFFF00000000FFFFFFFF00000000, 0x7FFFFFFF00000000FFFFFFFFFFFFFFFF]
    vals = special + [rng.getrandbits(127) for _ in range(64)]
    # limb patterns that maximise carries
    vals += [int.from_bytes(bytes(rng.choice([0, 0xFF]) for _ in range(16)), "little") & p for _ in range(64)]
    A = []; B = []
    for _ in range(4000):
        a = (rng.choice(vals), rng.choice(vals)); b = (rng.choice(vals), rng.choice(vals))
        A.append(O.f2_to_bytes_raw(a) if hasattr(O, "f2_to_bytes_raw") else (a[0].to_bytes(16, "little") + a[1].to_bytes(16, "little")))
        B.append(b[0].to_bytes(16, "little") + b[1].to_bytes(16, "little"))
    for op in ("mul", "add", "sub"):
        got = fp2_op(sim, op, A, B)
        for a, b, g in zip(A, B, got):
            assert g == O.row_fp2(op, a, b), (op, a.hex(), b.hex())
    for op in ("sqr", "neg", "conj"):
        got = fp2_op(sim, op, A)
        for a, g in zip(A, got):
            assert g == O.row_fp2(op, a), (op, a.hex())
    got = fp2_op(sim, "inv", A[:300])
    for a, g in zip(A[:300], got):
        assert g == O.row_fp2("inv", a)


def test_fp_mul_sqr_random_and_adversarial_vs_ints(sim):
    """GF(p) mul and the dedicated 10-product squaring (fp.cuh fp_sqr / fp_fold7) against Python ints (fields.py:42-51):
    edge values, carry-maximising limb patterns (any 128-bit input: the entry point reduces first), 100k random."""
    rng = random.Random(11)
    p = O.P127
    special = [0, 1, 2, p - 1, p, p + 1, p - 2, 1 << 126, (1 << 126) - 1, (1 << 127), (1 << 128) - 1, (1 << 64) - 1, (1 << 64) + 1, (1 << 96) - 1,
               0xFFFFFFFF, (1 << 127) - (1 << 32), (1 << 127) - (1 << 64) - 1, 0xFFFFFFFF00000000FFFFFFFF00000000, 0x7FFFFFFF00000000FFFFFFFFFFFFFFFF,
               0x7FFFFFFFFFFFFFFF0000000000000000, 0x7FFFFFFFFFFFFFFFFFFFFFFF00000000, 0x7FFFFFFF000000000000000000000000, 0x7FFFFFFFFFFFFFFF00000000FFFFFFFF]
    vals = list(special)
    for _ in range(4096):
        vals.append(int.from_bytes(bytes(rng.choice([0, 0xFF, 0x80, 0x7F, 0x01]) for _ in range(16)), "little"))
    vals += [rng.getrandbits(128) for _ in range(100000)]
    a = _rows([x.to_bytes(16, "little") for x in vals]); out = np.zeros_like(a)
    assert sim.sim_fp_row_op(FPOPS["sqr"], _p(a), None, _p(out), ctypes.c_size_t(len(vals))) == 0
    got = [int.from_bytes(bytes(out[16 * i:16 * i + 16]), "little") for i in range(len(vals))]
    assert got == [x * x % p for x in vals]
    ys = vals[1:] + vals[:1]
    b = _rows([y.to_bytes(16, "little") for y in ys])
    assert sim.sim_fp_row_op(FPOPS["mul"], _p(a), _p(b), _p(out), ctypes.c_size_t(len(vals))) == 0
    got = [int.from_bytes(bytes(out[16 * i:16 * i + 16]), "little") for i in range(len(vals))]
    assert got == [x * y % p for x, y in zip(vals, ys)]


def test_fp_inv_invsqrt_dbl_half(sim, golden):
    for which, key in ((0, "fp_inv"), (1, "fp_invsqrt")):
        rows = golden["fields"][key]
        a = _rows([H(r[0]) for r in rows]); out = np.zeros_like(a)
        sim.sim_fp_op(which, _p(a), _p(out), ctypes.c_size_t(len(rows)))
        assert [bytes(out[16 * i:16 * i + 16]).hex() for i in range(len(rows))] == [r[1] for r in rows]
    rng = random.Random(3)
    xs = [0, 1, O.P127 - 1, O.P127, 1 << 126] + [rng.getrandbits(127) for _ in range(200)]
    a = _rows([x.to_bytes(16, "little") for x in xs])
    for which, f in ((2, lambda x: 2 * x % O.P127), (3, lambda x: x * (1 << 126) % O.P127)):
        out = np.zeros_like(a)
        sim.sim_fp_op(which, _p(a), _p(out), ctypes.c_size_t(len(xs)))
        assert [int.from_bytes(bytes(out[16 * i:16 * i + 16]), "little") for i in range(len(xs))] == [f(x) for x in xs]


def test_codec_golden(sim, golden):
    c = golden["codec"]
    xy = _rows([H(r[0]) for r in c["encode"]]); enc = np.zeros(32 * len(c["encode"]), np.uint8)
    sim.sim_encode(_p(xy), _p(enc), ctypes.c_size_t(len(c["encode"])))
    assert [bytes(enc[32 * i:32 * i + 32]).hex() for i in range(len(c["encode"]))] == [r[1] for r in c["encode"]]
    e = _rows([H(r[0]) for r in c["decode"]]); n = len(c["decode"])
    out = np.zeros(64 * n, np.uint8); st = np.zeros(n, np.uint8)
    sim.sim_decode(_p(e), _p(out), _p(st), ctypes.c_size_t(n))
    for i, (enc_hex, want_st, want_xy) in enumerate(c["decode"]):
        assert (int(st[i]), bytes(out[64 * i:64 * i + 64]).hex()) == (want_st, want_xy), enc_hex


def test_recode_matches_reference_digits(sim):
    rng = random.Random(11)
    ks = [0, 1, 2, O.N - 1, O.N, O.N + 1, 2 * O.N, (1 << 256) - 1, ((1 << 256) // O.N) * O.N, ((1 << 256) // O.N) * O.N - 1]
    ks += [rng.getrandbits(256) for _ in range(2000)] + [rng.getrandbits(32) << 224 | rng.getrandbits(8) for _ in range(500)]
    for k in ks:
        kb = np.frombuffer(k.to_bytes(32, "little"), np.uint8).copy()
        idx = np.zeros(62, np.uint8); neg = np.zeros(62, np.uint8); red = np.zeros(32, np.uint8)
        sim.sim_recode(_p(kb), _p(idx), _p(neg), _p(red))
        ind, sgn = O.recode_windowed(k)
        r = k % O.N
        r += O.N if r % 2 == 0 else 0
        assert int.from_bytes(bytes(red), "little") == r
        assert ind[62] == 0 and sgn[62] == 1
        assert list(idx) == [ind[i] for i in range(61, -1, -1)]
        assert list(neg) == [1 - sgn[i] for i in range(61, -1, -1)]


def test_fixed_base_golden(sim, golden):
    rows = golden["mul"]["mul_base"]
    k = _rows([H(r[0]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8)
    sim.sim_fixed_base(0, _p(k), _p(out), None, ctypes.c_size_t(len(rows)))
    assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[1] for r in rows]
    rows = golden["mul"]["dh_base"]
    k = _rows([H(r[0]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8); st = np.zeros(len(rows), np.uint8)
    sim.sim_fixed_base(1, _p(k), _p(out), _p(st), ctypes.c_size_t(len(rows)))
    for i, (kk, want_st, want) in enumerate(rows):
        assert (int(st[i]), bytes(out[32 * i:32 * i + 32]).hex()) == (want_st, want), kk


def test_fixed_base_endo_golden(sim, golden):
    rows = golden["mul"]["mul_base"]
    k = _rows([H(r[0]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8)
    sim.sim_fixed_base(2, _p(k), _p(out), None, ctypes.c_size_t(len(rows)))
    assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[1] for r in rows]
    rows = golden["mul"]["dh_base"]
    k = _rows([H(r[0]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8); st = np.zeros(len(rows), np.uint8)
    sim.sim_fixed_base(3, _p(k), _p(out), _p(st), ctypes.c_size_t(len(rows)))
    for i, (kk, want_st, want) in enumerate(rows):
        assert (int(st[i]), bytes(out[32 * i:32 * i + 32]).hex()) == (want_st, want), kk


def test_fixed_base_comb_golden(sim, golden):
    """Per-digit tables (comb.cuh) give the reference's bytes for MUL_*(m, G, table) and DH_*(m, G, table=T392)."""
    rows = golden["mul"]["mul_base"]
    k = _rows([H(r[0]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8)
    sim.sim_comb(0, _p(k), _p(out), None, ctypes.c_size_t(len(rows)))
    assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[1] for r in rows]
    rows = golden["mul"]["dh_base"]
    k = _rows([H(r[0]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8); st = np.zeros(len(rows), np.uint8)
    sim.sim_comb(1, _p(k), _p(out), _p(st), ctypes.c_size_t(len(rows)))
    for i, (kk, want_st, want) in enumerate(rows):
        assert (int(st[i]), bytes(out[32 * i:32 * i + 32]).hex()) == (want_st, want), kk


def test_dh_golden(sim, golden):
    rows = golden["mul"]["dh"]
    k = _rows([H(r[0]) for r in rows]); e = _rows([H(r[1]) for r in rows]); n = len(rows)
    out = np.zeros(32 * n, np.uint8); st = np.zeros(n, np.uint8)
    sim.sim_dh(_p(k), _p(e), _p(out), _p(st), ctypes.c_size_t(n))
    for i, (kk, ee, want_st, want) in enumerate(rows):
        assert (int(st[i]), bytes(out[32 * i:32 * i + 32]).hex()) == (want_st, want), (kk, ee)
    rows = golden["mul"]["dh_affine"]
    k = _rows([H(r[0]) for r in rows]); xy = _rows([H(r[1]) for r in rows]); n = len(rows)
    out = np.zeros(64 * n, np.uint8); st = np.zeros(n, np.uint8)
    sim.sim_dh_affine(_p(k), _p(xy), _p(out), _p(st), ctypes.c_size_t(n))
    for i, (kk, pp, want_st, want) in enumerate(rows):
        assert (int(st[i]), bytes(out[64 * i:64 * i + 64]).hex()) == (want_st, want), (kk, pp)


def test_x25519_golden_and_rfc(sim, golden, x25519_kat):
    rows = golden["x25519"]["x25519"]
    k = _rows([H(r[0]) for r in rows]); u = _rows([H(r[1]) for r in rows]); out = np.zeros(32 * len(rows), np.uint8)
    sim.sim_x25519(_p(k), _p(u), _p(out), ctypes.c_size_t(len(rows)))
    assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[2] for r in rows]
    # the reference's own known answers (curve25519.py:96-107, :131-149), per row and through the shared inversion
    kat = x25519_kat
    k = _rows([H(r[0]) for r in kat]); u = _rows([H(r[1]) for r in kat])
    for fn in (lambda o: sim.sim_x25519(_p(k), _p(u), _p(o), ctypes.c_size_t(len(kat))),
               lambda o: sim.sim_x25519_batched(_p(k), _p(u), _p(o), ctypes.c_size_t(len(kat)), 16)):
        out = np.zeros(32 * len(kat), np.uint8); fn(out)
        assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(kat))] == [r[2] for r in kat]
    # RFC 7748 5.2 iteration vector (curve25519.py:104-124): 1 and 1000 iterations
    kk = uu = bytes([9] + [0] * 31)
    for i in range(1000):
        a = np.frombuffer(kk, np.uint8).copy(); b = np.frombuffer(uu, np.uint8).copy(); o = np.zeros(32, np.uint8)
        sim.sim_x25519(_p(a), _p(b), _p(o), ctypes.c_size_t(1))
        kk, uu = bytes(o), kk
        if i == 0:
            assert kk.hex() == "422c8e7a6227d7bca1350b3e2bb7279f7897b87bb6854b783c60e80311ae3079"
    assert kk.hex() == "684cf59ba83309552800ef566f2f4d3c1c3887c49360e3875f2eb94d99532c51"


def test_endo_pieces_golden(sim, golden):
    e = golden["endo"]
    for which, key in ((0, "phi"), (1, "psi")):
        rows = e[key]
        xy = _rows([H(r[0]) for r in rows]); out = np.zeros(64 * len(rows), np.uint8)
        sim.sim_endo_map(which, _p(xy), _p(out), ctypes.c_size_t(len(rows)))
        assert [bytes(out[64 * i:64 * i + 64]).hex() for i in range(len(rows))] == [r[1] for r in rows], key
    for (k, v), (v2, s, d) in zip(e["decompose"], e["recode"]):
        assert v == v2
        kb = np.frombuffer(H(k), np.uint8).copy()
        vv = np.zeros(4, np.uint64); idx = np.zeros(65, np.uint8); sg = np.zeros(65, np.uint8)
        sim.sim_endo_scalar(_p(kb), _p(vv), _p(idx), _p(sg))
        assert [int(x) for x in vv] == v, k
        assert "".join(str(int(x)) for x in sg) == s and "".join(str(int(x)) for x in idx) == d, k


def test_endo_scalar_random_vs_oracle(sim):
    rng = random.Random(21)
    for _ in range(3000):
        k = rng.getrandbits(256)
        kb = np.frombuffer(k.to_bytes(32, "little"), np.uint8).copy()
        vv = np.zeros(4, np.uint64); idx = np.zeros(65, np.uint8); sg = np.zeros(65, np.uint8)
        sim.sim_endo_scalar(_p(kb), _p(vv), _p(idx), _p(sg))
        v = O.decompose(k)
        assert [int(x) for x in vv] == v
        s, d = O.recode_endo(v)
        assert list(sg) == s and list(idx) == d


def test_dh_endo_golden(sim, golden):
    rows = golden["mul"]["dh"]
    k = _rows([H(r[0]) for r in rows]); e = _rows([H(r[1]) for r in rows]); n = len(rows)
    out = np.zeros(32 * n, np.uint8); st = np.zeros(n, np.uint8)
    sim.sim_dh_endo(_p(k), _p(e), _p(out), _p(st), ctypes.c_size_t(n))
    for i, (kk, ee, want_st, want) in enumerate(rows):
        assert (int(st[i]), bytes(out[32 * i:32 * i + 32]).hex()) == (want_st, want), (kk, ee)


def test_baseline_config1_sample(sim, golden):
    """BASELINE.json configs[0] on the instruction-level simulation of the device code (every 16th row, all three fixed-base
    algorithms of the device: windowed table, endomorphism table, per-digit comb)."""
    k = np.random.default_rng(1).integers(0, 256, (1024, 32), np.uint8)[::16].copy()
    want = golden["cfg1"]["out"][::16]
    n = len(k)
    for fn, args in (("sim_fixed_base", (1,)), ("sim_fixed_base", (3,)), ("sim_comb", (1,))):       # bit 0 = dh, bit 1 = endo
        out = np.zeros((n, 32), np.uint8); st = np.zeros(n, np.uint8)
        assert getattr(sim, fn)(*args, _p(k), _p(out), _p(st), ctypes.c_size_t(n)) == 0
        assert not st.any() and [bytes(r).hex() for r in out] == want, (fn, args)


def test_decode_spec_opt_in(sim, golden):
    rows = [r for r in golden["codec"]["decode"]]
    low = [O.encode(x, y) for x, y in (((0, 0), (1, 0)), ((0, 0), (O.P127 - 1, 0)), ((0, 1), (0, 0)), ((0, O.P127 - 1), (0, 0)))]
    enc = _rows([H(r[0]) for r in rows] + low)
    n = len(rows) + len(low)
    xy = np.zeros(64 * n, np.uint8); st = np.zeros(n, np.uint8)
    assert sim.sim_decode_spec(_p(enc), _p(xy), _p(st), ctypes.c_size_t(n)) == 0
    want = [O.row_decode(bytes(enc[32 * i:32 * i + 32]), spec=True) for i in range(n)]
    assert [(bytes(xy[64 * i:64 * i + 64]), int(st[i])) for i in range(n)] == want
    assert not st[-4:].any() and 3 not in set(int(s) for s in st)


def test_adversarial_grid_vs_c_oracle(sim):
    """Carry chains, Mersenne folds, recoding and decoding of the DEVICE code (instruction-level simulation) on limb patterns
    built to break them (tests/adversarial.py), against the C oracle: GF(p^2) ops on all-ones / boundary limbs and
    non-canonical inputs, and whole Diffie-Hellman rows (both algorithms) on special scalars x valid and invalid points."""
    import adversarial as A
    from oracle import c_oracle as C
    a, b = A.fp2_grid()
    n = len(a)
    for op in ("mul", "add", "sub", "sqr", "inv"):
        out = np.zeros_like(a)
        assert sim.sim_fp2_op(OPS[op], _p(a), _p(b) if op in ("mul", "add", "sub") else None, _p(out), ctypes.c_size_t(n)) == 0
        assert (out == C.fp2(op, a, b if op in ("mul", "add", "sub") else None)).all(), op
    k, enc = A.grid()
    n = len(k)
    want, wst = C.dh(k, enc)
    assert set(int(x) for x in wst) >= {0, 4, 5}
    for fn in ("sim_dh", "sim_dh_endo"):
        out = np.zeros((n, 32), np.uint8); st = np.zeros(n, np.uint8)
        assert getattr(sim, fn)(_p(k), _p(enc), _p(out), _p(st), ctypes.c_size_t(n)) == 0
        assert (st == wst).all() and (out == want).all(), fn


def _sim_rows(sim, fn, k, pt, width):
    n = len(k)
    out = np.full((n, width), 0xEE, np.uint8); st = np.full(n, 0xEE, np.uint8)
    assert getattr(sim, fn)(_p(k), _p(pt), _p(out), _p(st), ctypes.c_size_t(n)) == 0
    return out, st


def test_torsion_grid_vs_c_oracle(sim):
    """tests/torsion.py: the 392 points of the 392-torsion subgroup and prime-order points shifted by each of them, through the
    DEVICE DH code (both algorithms, encoded and affine entry points).  DH_core clears the cofactor first, so a pure torsion
    point gives the neutral point (status 5; 3 where decode stops at the reference's t == 0 quirk, i.e. the points of order
    1, 2 and 4) with a zero-filled row, and DH(k, P + T) == DH(k, P) for every T."""
    import torsion
    from oracle import c_oracle as C
    for affine, (k, pt, same) in ((False, torsion.grid()), (True, torsion.affine_grid())):
        want, wst = (C.dh_affine if affine else C.dh)(k, pt)
        tors = same < 0
        if affine:
            assert (wst[tors] == 5).all()
        else:
            quirk = np.array([O.decode_status(bytes(e))[0] == O.ST_QUIRK_T0 for e in pt])
            assert quirk.sum() == 4 * 3 and (quirk <= tors).all()                        # O, (0, -1), (+-i, 0), three scalars each
            assert (wst[quirk] == 3).all() and (wst[tors & ~quirk] == 5).all()
        assert not want[tors].any()
        assert (wst[~tors] == 0).all() and (want[~tors] == want[same[~tors]]).all()
        for fn in ("sim_dh_endo", "sim_dh") if not affine else ("sim_dh_endo_affine", "sim_dh_affine"):
            out, st = _sim_rows(sim, fn, k, pt, 64 if affine else 32)
            assert (st == wst).all() and (out == want).all(), fn


def test_torsion_grid_vs_plain_group_law(sim):
    """DH rows of the device code (simulation) against [392 k]A computed with the plain affine group law of tests/torsion.py,
    which shares no formula or recoding with the oracle: 32 pure torsion rows and 32 shifted rows of each grid."""
    import torsion
    rng = random.Random(392)
    for affine, (k, pt, same) in ((False, torsion.grid()), (True, torsion.affine_grid())):
        tors = np.flatnonzero(same < 0)
        rows = rng.sample(list(tors), 32) + rng.sample(list(np.flatnonzero(same >= 0)), 32)
        for fn in ("sim_dh_endo", "sim_dh") if not affine else ("sim_dh_endo_affine", "sim_dh_affine"):
            out, st = _sim_rows(sim, fn, k[rows], pt[rows], 64 if affine else 32)
            for i, r in enumerate(rows):
                if affine:
                    ws, A = O.ST_OK, O.xy_from_bytes(pt[r])
                else:
                    ws, A = O.decode_status(bytes(pt[r]))
                Q = torsion.dh_plain(int.from_bytes(bytes(k[r]), "little"), A) if ws == O.ST_OK else None
                if ws == O.ST_OK:
                    ws = O.ST_OK if Q is not None else O.ST_NEUTRAL
                w = bytes(64 if affine else 32) if Q is None else (torsion.xy(Q) if affine else torsion.enc(Q))
                assert (int(st[i]), bytes(out[i])) == (ws, w), (fn, r)
                assert (Q is None) == (r in tors)


def test_fixed_base_vs_plain_group_law(sim):
    """[k]G (MUL_windowed, MUL_endo, per-digit comb) and [392 k]G with the neutral check (the DH_base variants) of the device
    code against the plain affine group law of tests/torsion.py, on special and random scalars."""
    import adversarial
    import torsion
    rng = random.Random(393)
    ks = adversarial.special_scalars()
    ks = rng.sample(ks, 40) + [0, O.N, 2 * O.N] + [rng.getrandbits(256) for _ in range(21)]
    k = _rows([x.to_bytes(32, "little") for x in ks]).reshape(-1, 32)
    G = (O.GX, O.GY)
    want_mul = [torsion.enc(torsion.mul(x % O.N, G)) for x in ks]
    want_dh = [(5, bytes(32)) if Q is None else (0, torsion.enc(Q)) for Q in (torsion.dh_plain(x, G) for x in ks)]
    assert sum(w[0] == 5 for w in want_dh) == sum(x % O.N == 0 for x in ks) >= 3
    n = len(ks)
    for fn, mode in (("sim_fixed_base", 0), ("sim_fixed_base", 2), ("sim_comb", 0), ("sim_fixed_base", 1), ("sim_fixed_base", 3), ("sim_comb", 1)):
        out = np.full((n, 32), 0xEE, np.uint8); st = np.full(n, 0xEE, np.uint8)
        assert getattr(sim, fn)(mode, _p(k), _p(out), _p(st), ctypes.c_size_t(n)) == 0
        if mode & 1:
            assert [(int(s), bytes(o)) for s, o in zip(st, out)] == want_dh, (fn, mode)
        else:
            assert [bytes(o) for o in out] == want_mul, (fn, mode)


def test_x25519_special_values_vs_oracle(sim):
    """The device X25519 code (simulation) on special u coordinates x special scalars and 200 random rows vs the oracle."""
    rng = random.Random(91)
    p = (1 << 255) - 19
    us = [0, 1, 2, 9, p - 1, p, p + 1, (1 << 255) - 1, (1 << 256) - 1, 1 << 255, (1 << 254) + 7,
          325606250916557431795983626356110631294008115727848805560023387167927233504,
          39382357235489614581723060781553021112529911719440698176882885853963445705823,
          int("ffffffff00000000" * 4, 16), int("00000000ffffffff" * 4, 16)]
    ks = [0, 1, 8, (1 << 254), (1 << 255) - 1, (1 << 256) - 1, int("a5" * 32, 16), int("0f" * 32, 16)]
    kk = [int(a).to_bytes(32, "little") for a in ks for _ in us] + [rng.getrandbits(256).to_bytes(32, "little") for _ in range(200)]
    uu = [int(b).to_bytes(32, "little") for _ in ks for b in us] + [rng.getrandbits(256).to_bytes(32, "little") for _ in range(200)]
    k = _rows(kk); u = _rows(uu); out = np.zeros(32 * len(kk), np.uint8)
    sim.sim_x25519(_p(k), _p(u), _p(out), ctypes.c_size_t(len(kk)))
    assert [bytes(out[32 * i:32 * i + 32]) for i in range(len(kk))] == [O.x25519(a, b) for a, b in zip(kk, uu)]


def test_select_and_fp2_invsqrt_golden(sim, golden):
    """rows.cuh row_select / row_fp2_invsqrt against vectors produced by the reference's GFp.select, GFp2.select, GFp2.invsqrt."""
    g = golden["select"]
    for key, halves in (("fp_select", 1), ("fp2_select", 2)):
        rows = g[key]
        c = np.array([r[0] for r in rows], np.uint8)
        x = _rows([H(r[1]) for r in rows]); y = _rows([H(r[2]) for r in rows]); out = np.zeros_like(x)
        assert sim.sim_select(halves, _p(c), _p(x), _p(y), _p(out), ctypes.c_size_t(len(rows))) == 0
        w = 16 * halves
        assert [bytes(out[w * i:w * i + w]).hex() for i in range(len(rows))] == [r[3] for r in rows]
    rows = g["fp2_invsqrt"]
    a = _rows([H(r[0]) for r in rows]); out = np.zeros_like(a)
    assert sim.sim_fp2_invsqrt(_p(a), _p(out), ctypes.c_size_t(len(rows))) == 0
    assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[1] for r in rows]
    # random rows against the oracle, including the GF(p) branch
    rng = random.Random(21)
    A = [(rng.getrandbits(128).to_bytes(16, "little") + (b"\0" * 16 if i % 5 == 0 else rng.getrandbits(128).to_bytes(16, "little"))) for i in range(400)]
    a = _rows(A); out = np.zeros_like(a)
    sim.sim_fp2_invsqrt(_p(a), _p(out), ctypes.c_size_t(len(A)))
    assert [bytes(out[32 * i:32 * i + 32]) for i in range(len(A))] == [O.row_fp2("invsqrt", x) for x in A]


@pytest.mark.parametrize("rows_per_thread", [1, 4, 16, 32])
def test_batched_inversion_with_zero_rows_in_every_position(sim, rows_per_thread):
    """batchinv.cuh (k_fp2_inv_batched): zeros, p (an alias of zero), ones and random values mixed inside the groups that share
    one inversion, ragged batch sizes; inv(0) = 0 as in fields.py:194-199."""
    rng = random.Random(31 + rows_per_thread)
    p = O.P127
    for n in (1, 2, 63, 64, 65, 1000, 64 * rows_per_thread + 1):
        A = []
        for i in range(n):
            r = rng.random()
            if r < 0.15:
                a = (rng.choice([0, p, 1 << 127]) if rng.random() < 0.7 else 0, rng.choice([0, p]))     # zero in every disguise (2^127 = 1: not zero)
            elif r < 0.25:
                a = (1, 0)
            else:
                a = (rng.getrandbits(128), rng.getrandbits(128))
            A.append(a[0].to_bytes(16, "little") + a[1].to_bytes(16, "little"))
        a = _rows(A); out = np.full_like(a, 0xEE)
        assert sim.sim_fp2_inv_batched(_p(a), _p(out), ctypes.c_size_t(n), rows_per_thread) == 0
        got = [bytes(out[32 * i:32 * i + 32]) for i in range(n)]
        assert got == [O.row_fp2("inv", x) for x in A], (n, rows_per_thread)


def test_finish_kernel_mixed_groups(sim):
    """batchinv.cuh FinishIO (k_dh_finish): projective rows with Z = 0 (also as p in either half) / failed status / the neutral
    point mixed with good rows in one shared inversion; compared with the per-row R1toAffine + neutral check + encode of the
    oracle.  A zero Z that entered the shared product would zero the results of every row in its group."""
    rng = random.Random(41)
    p = O.P127
    G = (O.GX, O.GY)
    pts = []
    P = O.affine_to_r1(*G)
    for _ in range(40):
        P = O.dbl(P)
        pts.append(O.r1_to_affine(P))
    n = 333
    rows, st_in, want, wst = [], [], [], []
    for i in range(n):
        r = rng.random()
        x, y = pts[i % len(pts)]
        lam = (rng.getrandbits(127) % p or 1, rng.getrandbits(127) % p)
        X, Y, Z = O.f2_mul(x, lam), O.f2_mul(y, lam), lam
        st = 0
        if r < 0.1:
            X, Y, Z, st = (rng.getrandbits(127), 5), (7, rng.getrandbits(127)), (0, 0), 4          # failed validation: garbage with Z = 0
        elif r < 0.2:
            st = rng.choice([1, 2, 3, 4])                                                          # failed validation, harmless coordinates
        elif r < 0.3:
            X, Y, Z = rng.choice([(0, 0), (p, 0), (p, p)]), lam, lam                              # the neutral point (0, 1), x = 0 in any form
        elif r < 0.4:                                                                              # failed validation, Z a non-canonical zero:
            Z, st = rng.choice([(p, 0), (0, p), (p, p)]), rng.choice([1, 2, 3, 4])                 # "zero is 0 or p" (fp.cuh fp_is_zero)
        rows.append(b"".join(v.to_bytes(16, "little") for v in (X[0], X[1], Y[0], Y[1], Z[0], Z[1])))
        st_in.append(st)
        if st != 0:
            want.append(bytes(32)); wst.append(st)
        elif (X[0] % p, X[1] % p) == (0, 0) and Y == Z:
            want.append(bytes(32)); wst.append(5)
        else:
            zi = O.f2_inv(Z)
            want.append(bytes(O.encode(O.f2_mul(X, zi), O.f2_mul(Y, zi)))); wst.append(0)
    for rpt in (1, 4, 16):
        a = _rows(rows); s_in = np.array(st_in, np.uint8); out = np.full(32 * n, 0xEE, np.uint8); st = np.full(n, 0xEE, np.uint8)
        assert sim.sim_finish_rows(_p(a), _p(s_in), _p(out), _p(st), ctypes.c_size_t(n), rpt, 1) == 0
        assert [bytes(out[32 * i:32 * i + 32]) for i in range(n)] == want and list(st) == wst


def test_x25519_shared_inversion(sim, golden):
    """x25519.cuh X25519FinIO: the RFC / golden rows through the batched finish (one z^(p-2) chain per 16 rows), u = 0 rows (z2 = 0)
    mixed in."""
    rows = golden["x25519"]["x25519"]
    k = _rows([H(r[0]) for r in rows]); u = _rows([H(r[1]) for r in rows]); out = np.zeros_like(k)
    for rpt in (1, 16):
        assert sim.sim_x25519_batched(_p(k), _p(u), _p(out), ctypes.c_size_t(len(rows)), rpt) == 0
        assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[2] for r in rows]


F25OP = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4}


def test_gfp25519_field_ops_golden_and_batched_inversion(sim, golden):
    """x25519.cuh row_f25_op / F25InvIO against vectors produced by the reference's GFp25519.add/sub/mul/sqr/inv (unreduced operands,
    p, 2p, 2^256 - 1 among them); the inversion also through the shared chain with zeros (0, p, 2p) in every group size."""
    g = golden["f25519"]
    for op in ("add", "sub", "mul"):
        rows = g[op]
        a = _rows([H(r[0]) for r in rows]); b = _rows([H(r[1]) for r in rows]); out = np.zeros_like(a)
        assert sim.sim_f25_op(F25OP[op], _p(a), _p(b), _p(out), ctypes.c_size_t(len(rows))) == 0
        assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[2] for r in rows], op
    for op in ("sqr", "inv"):
        rows = g[op]
        a = _rows([H(r[0]) for r in rows]); out = np.zeros_like(a)
        assert sim.sim_f25_op(F25OP[op], _p(a), None, _p(out), ctypes.c_size_t(len(rows))) == 0
        assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[1] for r in rows], op
    rows = g["inv"]
    a = _rows([H(r[0]) for r in rows])
    for rpt in (1, 4, 16, 32):
        out = np.full_like(a, 0xEE)
        assert sim.sim_f25_inv_batched(_p(a), _p(out), ctypes.c_size_t(len(rows)), rpt) == 0
        assert [bytes(out[32 * i:32 * i + 32]).hex() for i in range(len(rows))] == [r[1] for r in rows], rpt
    rng = random.Random(2519)
    q = O.P25519
    for n in (1, 63, 65, 1000):
        A = [rng.choice([0, q, 2 * q, 1, q - 1, rng.getrandbits(256), rng.getrandbits(256)]).to_bytes(32, "little") for _ in range(n)]
        a = _rows(A); out = np.full_like(a, 0xEE)
        assert sim.sim_f25_inv_batched(_p(a), _p(out), ctypes.c_size_t(n), 16) == 0
        assert [bytes(out[32 * i:32 * i + 32]) for i in range(n)] == [O.row_f25519("inv", x) for x in A]
