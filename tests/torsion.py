"""Points with a small-order component, shared by the CPU simulation test and the GPU tests: the 392 points of the
392-torsion subgroup of Curve4Q (orders 1, 2, 4, 7, 8, 14, 28, 56), prime-order points shifted by them, and a plain affine
group law in Python ints to check scalar multiplications against.

DH_core clears the cofactor ([392]P) before the ladder, so a pure torsion point must give the neutral point (status 5, or 3
where decode stops first at the reference's t == 0 quirk) and DH(k, P + T) must equal DH(k, P) byte for byte.  The group
law here shares no code with the oracle's point formulas or recodings: only the curve constants and encode / decode_status
are taken from it."""
import random

import numpy as np

from oracle import c_oracle as C
from oracle import fourq_oracle as O

P = O.P127
D = O.D
N = O.N
COFACTOR = 392
NEUTRAL = ((0, 0), (1, 0))
DIVISORS = [d for d in range(1, COFACTOR + 1) if COFACTOR % d == 0]


# ---------------------------------------------------------------- GF(p^2) = GF(p)[i] / (i^2 + 1) and the affine group law

def _f2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % P, (a[0] * b[1] + a[1] * b[0]) % P)


def _f2_inv(a):
    n = pow((a[0] * a[0] + a[1] * a[1]) % P, P - 2, P)
    return (a[0] * n % P, -a[1] * n % P)


def add(A, B):
    """Affine addition on -x^2 + y^2 = 1 + d x^2 y^2: x3 = (x1 y2 + y1 x2) / (1 + t), y3 = (y1 y2 + x1 x2) / (1 - t) with
    t = d x1 x2 y1 y2.  Complete, since d is not a square in GF(p^2): no denominator is ever zero."""
    (x1, y1), (x2, y2) = A, B
    xx, yy = _f2_mul(x1, x2), _f2_mul(y1, y2)
    t = _f2_mul(D, _f2_mul(xx, yy))
    xy, yx = _f2_mul(x1, y2), _f2_mul(y1, x2)
    plus, minus = ((1 + t[0]) % P, t[1]), ((1 - t[0]) % P, -t[1] % P)
    inv = _f2_inv(_f2_mul(plus, minus))                        # one inversion for both denominators
    x3 = _f2_mul(((xy[0] + yx[0]) % P, (xy[1] + yx[1]) % P), _f2_mul(inv, minus))
    y3 = _f2_mul(((yy[0] + xx[0]) % P, (yy[1] + xx[1]) % P), _f2_mul(inv, plus))
    return x3, y3


def mul(k, A):
    """[k]A by double-and-add, k >= 0."""
    R = NEUTRAL
    for b in bin(k)[2:]:
        R = add(R, R)
        if b == "1":
            R = add(R, A)
    return R


def on_curve(A):
    (x, y) = A
    x2, y2 = _f2_mul(x, x), _f2_mul(y, y)
    lhs = ((y2[0] - x2[0]) % P, (y2[1] - x2[1]) % P)
    r = _f2_mul(D, _f2_mul(x2, y2))
    return lhs == ((1 + r[0]) % P, r[1])


def order(T):
    """Order of a point of the 392-torsion subgroup."""
    return next(d for d in DIVISORS if mul(d, T) == NEUTRAL)


def enc(A):
    return O.encode(A[0], A[1])


def xy(A):
    return b"".join(int(v).to_bytes(16, "little") for v in (A[0][0], A[0][1], A[1][0], A[1][1]))


def dh_plain(k, A):
    """DH_core by definition: [392 k]A, or None where it is the neutral point."""
    Q = mul(COFACTOR * (k % N), A)
    return None if Q == NEUTRAL else Q


# ---------------------------------------------------------------- the 392-torsion subgroup

def _decodable_points(seed):
    rng = random.Random(seed)
    while True:
        e = bytearray(rng.getrandbits(256).to_bytes(32, "little"))
        e[15] &= 0x7F
        st, A = O.decode_status(bytes(e))
        if st == O.ST_OK:
            yield A


_TORSION = None


def torsion_points():
    """[(T, order)]: all 392 points T with [392]T = O, sorted by order and coordinates.  Built from [N]R for a fixed-seed
    sequence of decodable points R (each has a random torsion component), closing the set under addition until it stops
    growing."""
    global _TORSION
    if _TORSION is None:
        pts, gens = {NEUTRAL}, []
        src = _decodable_points(392)
        for _ in range(16):
            gens.append(mul(N, next(src)))
            new = set(pts)
            while new:                                         # the closure of pts under adding any generator
                new = {add(a, g) for a in new for g in gens} - pts
                pts |= new
            if len(pts) == COFACTOR:
                break
        assert len(pts) == COFACTOR, len(pts)
        assert all(on_curve(T) and mul(COFACTOR, T) == NEUTRAL for T in pts)
        _TORSION = sorted(((T, order(T)) for T in pts), key=lambda r: (r[1], r[0]))
    return _TORSION


def shifted(A, T):
    """A + T in affine form and its encoding."""
    S = add(A, T)
    return S, enc(S)


def prime_order_points(n, seed=7):
    """n points of the prime-order subgroup, [k]G for seeded k, as (encoding, affine point)."""
    ks = np.random.default_rng(seed).integers(0, 256, (n, 32), np.uint8)
    out = []
    for e in C.mul_base(ks):
        st, A = O.decode_status(bytes(e))
        assert st == O.ST_OK
        out.append((bytes(e), A))
    return out


def scalars(seed=392):
    """adversarial.special_scalars() thinned to 8 (0, 1, N - 1, N, N + 1, 2^256 - 1, the largest multiple of N below 2^256 and
    one from the middle of the list), plus 3 random ones."""
    import adversarial
    s = adversarial.special_scalars()
    thin = [0, 1, N - 1, N, N + 1, s[len(s) // 2], (1 << 256) - 1, ((1 << 256) // N) * N]
    assert all(x in s for x in thin)
    rng = random.Random(seed)
    return thin + [rng.getrandbits(256) for _ in range(3)]


def _rows(lst):
    return np.frombuffer(b"".join(lst), np.uint8).reshape(len(lst), -1).copy()


def _grid(point_bytes, per_torsion=3, npoints=3, seed=392):
    """Rows of (k, point, same_as): every torsion point against `per_torsion` scalars (rotating through scalars(), so every
    scalar meets every order), then for each of `npoints` prime-order P one scalar k (1, N - 1, then random ones) against P
    and against P + T for every T.
    same_as[i] = -1 for a pure torsion row, else the index of the (k, P) row whose result row i must equal."""
    ks = [int(x).to_bytes(32, "little") for x in scalars(seed)]
    tors = torsion_points()
    kk, pp, same = [], [], []
    for i, (T, _) in enumerate(tors):
        for j in range(per_torsion):
            kk.append(ks[(i + j * 5) % len(ks)]); pp.append(point_bytes(T)); same.append(-1)
    rng = random.Random(seed)
    for j, (e, A) in enumerate(prime_order_points(npoints, seed)):
        k = int((1, N - 1)[j] if j < 2 else rng.getrandbits(256)).to_bytes(32, "little")
        base = len(kk)
        kk.append(k); pp.append(point_bytes(A)); same.append(base)
        for T, _ in tors:
            kk.append(k); pp.append(point_bytes(add(A, T))); same.append(base)
    return _rows(kk), _rows(pp), np.array(same, np.int64)


_GRIDS = {}


def grid():
    """(k[n,32], enc[n,32], same_as[n]) for the encoded-point entry points (see _grid), about 2,300 rows."""
    if "enc" not in _GRIDS:
        _GRIDS["enc"] = _grid(enc)
    return _GRIDS["enc"]


def affine_grid():
    """(k[n,32], xy[n,64], same_as[n]): the same points as 64-byte x | y rows for the affine entry points.  These reach the
    points of order 1, 2 and 4, whose encodings decode rejects with status 3 before DH runs."""
    if "xy" not in _GRIDS:
        _GRIDS["xy"] = _grid(xy)
    return _GRIDS["xy"]
