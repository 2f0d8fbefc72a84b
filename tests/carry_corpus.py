"""The carry corpus: deterministic rows, per GPU entry point, that drive the carry chains of the device arithmetic (fp.cuh,
x25519.cuh, scalar.cuh, endo.cuh) both ways.  tests/test_carry.py runs them through the carry sanitizer of the CPU simulation
and checks that every carry primitive's call site produced and consumed carries of 0 and 1; tests/test_gpu_carry.py runs the
same rows through the GPU entry points.

Sources: the shared adversarial values (tests/adversarial.py), targeted constructions for carries that random rows almost
never produce (named below, next to the chain they reach), and a small seeded search for the rest.  Each row set is named
after its fq_dev_run op (fourq_b200/_lib.py DEVOP) and holds that op's input arrays."""
import random

import numpy as np

import adversarial
from oracle import c_oracle as C
from oracle import fourq_oracle as O

P = O.P127
Q = O.P25519
M32 = 0xFFFFFFFF


def _u(vals, width):
    return np.stack([np.frombuffer(int(v).to_bytes(width, "little"), np.uint8) for v in vals]).copy()


def _limbs(a0, a1, a2, a3):
    return a0 | a1 << 32 | a2 << 64 | a3 << 96


# ---------------------------------------------------------------- GF(p)

def fp_sqr_fold7():
    """fp_fold7's second pass carries the +1 out of limb 2 into limb 3 only when the first pass leaves limbs 0..2 all ones and bit
    127 set: a = p - 2^48 gives a^2 = 2^96 (mod p) on the way.  Its multiples by small powers of two land on the same chain."""
    a = P - (1 << 48)
    return [a] + [a * (1 << s) % P for s in range(1, 32)] + [P - (1 << s) for s in range(40, 64)]


def fp_sqr_even_catches(rng, count=48):
    """fp_sqr's even lattice: the catch E4 = addc_cc(E4, 0) carries out when E4 = 2^32 - 1 after its first chain and the W^2 chain of
    the second carries in.  With a2's top bit set d3 = 2 a3 + 1 is odd, so a1 = (2^32 - 1 - lo(a2^2) - c) / d3 mod 2^32 sets E4.
    E5 carries on when the W^4 pair E5:E4 = a1 d3 + a2^2 + c is 2^64 - 1: a2 close to 2^32 leaves a small rest 2^64 - 1 - c - a2^2 to
    split as a1 * d3 with d3 odd."""
    out = []
    for _ in range(count):
        a0, a2, a3 = rng.getrandbits(32), rng.getrandbits(32) | 1 << 31, rng.getrandbits(31)
        d3 = (a3 << 1 | a2 >> 31) & M32
        for c in (0, 1):
            a1 = (M32 - (a2 * a2 & M32) - c) * pow(d3, -1, 1 << 32) & M32
            out.append(_limbs(a0, a1, a2, a3))
    for a2 in range(M32, M32 - 4096, -1):
        for c in (0, 1):
            rest = (1 << 64) - 1 - c - a2 * a2
            for d3 in (M32, M32 - 2, M32 - 4, 3, 5, 7, 9, 15, 17, 255, 257, 65535, 65537):
                if rest % d3 == 0 and rest // d3 <= M32 and (d3 & 1) == (a2 >> 31):
                    a1, a3 = rest // d3, d3 >> 1
                    out += [_limbs(rng.getrandbits(32), a1, a2, a3) for _ in range(4)]
        if len(out) >= 4 * count:
            break
    return [x % (1 << 128) for x in out]


def fp_values(rng):
    vals = set(adversarial.special_fp_values())
    vals |= {P + 1, 1 << 127, (1 << 128) - 1, (1 << 128) - 2, (1 << 127) - 1 + (1 << 127), 0xFFFFFFFF00000000FFFFFFFF00000000,
             0x7FFFFFFF00000000FFFFFFFFFFFFFFFF, 0x7FFFFFFFFFFFFFFF0000000000000000, 0x7FFFFFFFFFFFFFFFFFFFFFFF00000000,
             0x7FFFFFFF000000000000000000000000, 0x7FFFFFFFFFFFFFFF00000000FFFFFFFF}
    vals |= {v | 1 << 127 for v in list(vals) if v < (1 << 127)}                      # non-canonical inputs: the entry points reduce
    pats = [int.from_bytes(bytes(rng.choice([0, 0xFF, 0x80, 0x7F, 0x01]) for _ in range(16)), "little") for _ in range(256)]
    return sorted(vals) + pats + [rng.getrandbits(128) for _ in range(128)]


def fp_pairs(rng, vals, n):
    """Operand pairs for add / sub / mul: every value against its neighbours, against p - itself, and random pairs."""
    a, b = [], []
    for i, x in enumerate(vals):
        for y in (vals[(i + 1) % len(vals)], (P - x) % (1 << 128), (x + 1) % (1 << 128), ((1 << 128) - 1) ^ x):
            a.append(x); b.append(y)
    while len(a) < n:
        a.append(rng.choice(vals)); b.append(rng.choice(vals))
    return a, b


# ---------------------------------------------------------------- GF(2^255 - 19)

def f25_values(rng):
    v = {0, 1, 2, 19, 37, 38, 39, Q - 1, Q, Q + 1, 2 * Q, 2 * Q + 1, 2 * Q + 37, (1 << 255) - 1, 1 << 255, (1 << 255) + 18,
         (1 << 256) - 1, (1 << 256) - 2, (1 << 256) - 38, (1 << 256) - 39, (1 << 256) - 19, 1 << 128, (1 << 64) - 1, 1 << 224,
         int("ff" * 16 + "00" * 16, 16), int("00" * 16 + "ff" * 16, 16), int("ffffffff00000000" * 4, 16), int("00000000ffffffff" * 4, 16)}
    for s in (32, 64, 96, 128, 160, 192, 224, 254):
        v |= {(1 << 256) - (1 << s), (1 << s) - 1}
    pats = [int.from_bytes(bytes(rng.choice([0, 0xFF, 0xFE, 0x80, 0x7F, 0x01]) for _ in range(32)), "little") for _ in range(128)]
    return sorted(v) + pats + [rng.getrandbits(256) for _ in range(64)]


def f25_add_sub_pairs(rng, vals):
    """f25_add wraps twice (fix_carry's second wrap) when a + b lands in [2^256 + 2^256 - 38, 2^257): operands near 2^256; f25_sub
    borrows twice when a - b + 2^256 < 38: b just above a."""
    a, b = [], []
    for x in vals:
        for y in (x, (1 << 256) - 1 - x, (1 << 256) - x + 37, x + 1, x + 37, (1 << 256) - 1, 0):
            a.append(x); b.append(y % (1 << 256))
    for d in range(0, 40):
        a += [(1 << 256) - 1 - d, d, (1 << 256) - 20 + d % 20]
        b += [(1 << 256) - 1 - (39 - d), d + 1 + d % 3, (1 << 256) - 1]
    for _ in range(512):
        x = rng.getrandbits(256)
        a += [x, x]; b += [(x + rng.randrange(1, 38)) % (1 << 256), ((1 << 256) - x + rng.randrange(0, 64)) % (1 << 256)]
    return a, b


# X25519 rows whose ladder reaches the carries of f25_mul_a24 (a * 121665): its chain carries only when lo(a_i 121665) lands within
# 121665 of 2^32, about once per 10^5 multiplications.  Found by a seeded search over random (k, u) (random.Random(25519), rows
# 2013, 2265, 2276, 2669, 2389, 2492, 2881 of 3000): the first four carry into t[8], the last three out of t[1].
X25519_SEARCHED = [
    (0xa633597894b24146841d8790c9273b539e47278a91913368ae0bd7e78835baf3, 0x641d6550c9b23d8694ec572c0d303e1833c19fc29215e6b16f95d55ce55cbb9d),
    (0xf6e9cfbd58353ae817770f97a56ce7b881dd4ba7a540deab00a345826901ed63, 0x8c6d5c48f6e6844912de4259cbe4613daaacc8a7302f63760abf8d4b15ef6770),
    (0x4c7fd3536d8596a99fd66a140aabee9c0e542e82d82297766589e556be5adc0a, 0xe42a7e906bd8625e832f3429c7fd2da4319f040c09f476125f99536704d798d8),
    (0x5a77dff3615e8e672e971ff4ed282f24186716545cde4b83842ef3cecf19d322, 0x718ad65129976b04e84e03b0cad643f034e09a43b4aab8f11f982f0d28ff79c7),
    (0x550c3765b8800807e86327f78f7afcca6fb29a9520b127d29604c3d2e38531, 0xce9ec4e4a4cf8dc31f9b28ecb5733793796b23a7e614f88f0a54e7c0a6a53985),
    (0x2cdbbd0bdca3591a5dd7070cf73868221571f35857196baf74b2b5d0128095b2, 0xea236cf23c0fd8be5d4dcb4a6fde4f189bef52e2983606b4eb5a5163cf7aa43d),
    (0x601558718d7f22500e612692b0b785dfd554ea34adc777a25c04763c7ced8dd3, 0xa927943239b15813cab13e3a53a675bef7a8744df34d09f5ce78b9d07b457386),
]


# ---------------------------------------------------------------- the row sets

class RowSet:
    """Rows of one fq_dev_run op (a key of fourq_b200._lib.DEVOP): ins = its input arrays (a, b, c as that op takes them)."""
    def __init__(self, name, op, ins):
        self.name, self.op, self.ins = name, op, [np.ascontiguousarray(x) for x in ins]

    @property
    def n(self):
        return self.ins[0].shape[0]


def build():
    rng = random.Random(0xCA77)
    sets = []
    fv = fp_values(rng)
    a, b = fp_pairs(rng, fv, 3000)
    A, B = _u(a, 16), _u(b, 16)
    sq = _u(fp_sqr_fold7() + fp_sqr_even_catches(rng) + fv, 16)
    for op in ("mul", "add", "sub"):
        sets.append(RowSet("fp_" + op, "fp_" + op, [A, B]))
    sets.append(RowSet("fp_sqr", "fp_sqr", [sq]))
    sets.append(RowSet("fp_neg", "fp_neg", [A]))
    sets.append(RowSet("fp_inv", "fp_inv", [_u(fv[:96], 16)]))
    sets.append(RowSet("fp_invsqrt", "fp_invsqrt", [_u(fv[:96], 16)]))
    # GF(p^2): the adversarial grid (every special value in both halves) plus the GF(p) targets as real and imaginary parts
    ga, gb = adversarial.fp2_grid()
    tg = fp_sqr_fold7() + fp_sqr_even_catches(random.Random(2))[:64]
    t2 = _u([x | y << 128 for x in tg for y in (0, tg[0], P - 1)], 32)
    fa = np.concatenate([ga, t2]); fb = np.roll(fa, 7, axis=0)
    for op in ("mul", "add", "sub"):
        sets.append(RowSet("fp2_" + op, "fp2_" + op, [fa, fb]))
    for op in ("sqr", "neg", "conj"):
        sets.append(RowSet("fp2_" + op, "fp2_" + op, [fa]))
    inv_rows = np.concatenate([_u([0, P, P << 128, P | P << 128], 32), fa[::9]])
    sets.append(RowSet("fp2_inv", "fp2_inv", [inv_rows]))
    sets.append(RowSet("fp2_invsqrt", "fp2_invsqrt", [np.concatenate([fa[::23], _u(tg[:16], 32)])]))
    sel = fa[::5]
    sets.append(RowSet("fp2_select", "fp2_select", [sel, np.roll(sel, 3, axis=0), np.resize(np.array([0, 1, 2, 0xFF], np.uint8), sel.shape[0])[:, None]]))
    # GF(2^255 - 19)
    qv = f25_values(rng)
    qa, qb = f25_add_sub_pairs(rng, qv)
    QA, QB = _u(qa, 32), _u(qb, 32)
    for op in ("add", "sub"):
        sets.append(RowSet("f25519_" + op, "f25519_" + op, [QA, QB]))
    pa = [x for x in qv for _ in range(4)]
    pb = [rng.choice(qv) for _ in pa]
    sets.append(RowSet("f25519_mul", "f25519_mul", [_u(pa, 32), _u(pb, 32)]))
    sets.append(RowSet("f25519_sqr", "f25519_sqr", [_u(qv, 32)]))
    sets.append(RowSet("f25519_inv", "f25519_inv", [_u(qv[:64], 32)]))
    # X25519: special u x special k
    us = [0, 1, 2, 9, Q - 1, Q, Q + 1, (1 << 255) - 1, (1 << 256) - 1, (1 << 255) + 18, int("ffffffff00000000" * 4, 16)]
    ks = [0, (1 << 256) - 1, int("a5" * 32, 16), rng.getrandbits(256)]
    xk = [k for k in ks for _ in us] + [k for k, _ in X25519_SEARCHED]
    xu = [u for _ in ks for u in us] + [u for _, u in X25519_SEARCHED]
    sets.append(RowSet("x25519", "x25519", [_u(xk, 32), _u(xu, 32)]))
    # decode: the adversarial encodings and the t == 0 / low-order / non-canonical ones
    _, enc = adversarial.grid()
    low = [O.encode(x, y) for x, y in (((0, 0), (1, 0)), ((0, 0), (P - 1, 0)), ((0, 1), (0, 0)), ((0, P - 1), (0, 0)))]
    dec = np.concatenate([np.unique(enc, axis=0), np.frombuffer(b"".join(low), np.uint8).reshape(-1, 32), _u([P, P << 128, (1 << 256) - 1], 32)])
    sets.append(RowSet("decode", "decode", [dec]))
    # scalars: scal_reduce_odd (MUL_windowed) and endo_mulhi_256 (MUL_endo, DH_endo)
    sk = adversarial.special_scalars()
    ks = _u(sk + [rng.getrandbits(256) for _ in range(8)], 32)
    sets.append(RowSet("mul_base", "mul_base", [ks]))
    sets.append(RowSet("mul_endo_base", "mul_endo_base", [ks]))
    G = O.encode(O.GX, O.GY)
    pk = np.tile(np.frombuffer(G, np.uint8), (12, 1))
    sets.append(RowSet("dh_endo", "dh_endo", [ks[:: max(1, len(ks) // 12)][:12], pk]))
    return sets


def _py(fn, *cols):
    return np.frombuffer(b"".join(fn(*[bytes(c[i]) for c in cols]) for i in range(cols[0].shape[0])), np.uint8).reshape(cols[0].shape[0], -1)


def reference(rs):
    """(out, status or None) of rs from the C oracle where it has the op, else the Python oracle."""
    op, ins = rs.op, rs.ins
    kind, _, name = op.partition("_")
    if op == "fp2_select":
        return _py(lambda x, y, c: O.row_select(c[0], x, y), *ins), None
    if op == "fp2_invsqrt":
        return _py(lambda x: O.row_fp2("invsqrt", x), ins[0]), None
    if kind == "fp2":
        return C.fp2(name, *ins), None
    if kind == "fp":
        return C.fp(name, *ins), None
    if kind == "f25519":
        return _py(lambda *x: O.row_f25519(name, *x), *ins), None
    if op == "x25519":
        return _py(O.x25519, *ins), None
    if op == "decode":
        return C.decode(ins[0])
    if op in ("mul_base", "mul_endo_base"):
        return C.mul_base(ins[0]), None
    if op == "dh_endo":
        return C.dh(*ins)
    raise AssertionError(op)
