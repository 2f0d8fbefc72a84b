"""Batched Curve4Q -- the counterpart of the reference's impl/curve4q.py entry points.

    reference (one element, Python ints)            here (N rows, numpy uint8)
    PointOnCurve((X, Y)) -> bool       :23-29       PointOnCurve(XY[N,64]) -> bool[N]
    encode(X, Y) -> bytearray(32)      :41-46       encode(XY[N,64]) -> B[N,32]
    decode(B) -> (x, y) or raises      :49-96       decode(B[N,32]) -> (XY[N,64], status[N])
    DH_windowed(m, P) -> affine Q      :464-465     DH_windowed(k[N,32], XY[N,64]) -> (XY[N,64], status[N])
    DH_endo(m, P) -> affine Q          :467-468     DH_endo(k[N,32], XY[N,64]) -> (XY[N,64], status[N])
    encode(DH_*(m, decode(B)))                      DH(k[N,32], B[N,32], algorithm=) -> (B[N,32], status[N])
    y of DH_*(m, decode(B))  (draft :707-714)       DH(k, B, y_only=True) -> (y[N,32], status[N])
    DH_*(m, G, table=T392)             :743-762     DH_base(k[N,32], algorithm=) -> (B[N,32], status[N])
    MUL_*(m, G, table=T) -> [m]G       :582-584     MUL_base(k[N,32], algorithm=) -> B[N,32]
    encode(DH_windowed(m, P)), one P                FixedBase(P).DH(k[N,32]) -> (B[N,32], status[N])
    encode(MUL_windowed(m, P)), one P  :188-235     FixedBase(P).MUL(k[N,32]) -> B[N,32]

algorithm = "windowed" runs MUL_windowed (curve4q.py:188-235), "endo" runs MUL_endo (curve4q.py:405-442); the results
are bit-identical (the reference asserts it, curve4q.py:706-762), "endo" needs about 1.8x fewer field multiplications
and is the default.  The fixed-base entry points DH_base / MUL_base also take algorithm = "comb" (their default): one
precomputed table per digit, 62 mixed additions and no doubling -- the fixed-base method the draft recommends for key
generation (draft-ladd-cfrg-4q.md:702-705, :727-729); same bytes again because the affine result is canonical.

Scalars are 32-byte little-endian unsigned rows (no clamping).  Exceptions of the reference become per-row status codes;
failed rows are zero-filled.  `strict=True` raises the reference's message for the first failing row instead.
decode() does not modify its argument (the reference clears bits in place, curve4q.py:56).
"""
import ctypes

import numpy as np

from . import _lib

DEFAULT_ALGORITHM = "endo"
_ALGS = ("windowed", "endo")


DEFAULT_BASE_ALGORITHM = "comb"
_BASE_ALGS = ("windowed", "endo", "comb")


def _alg(algorithm, base=False):
    a = (DEFAULT_BASE_ALGORITHM if base else DEFAULT_ALGORITHM) if algorithm is None else algorithm
    if a not in (_BASE_ALGS if base else _ALGS):
        raise ValueError("algorithm must be one of %r" % ((_BASE_ALGS if base else _ALGS),))
    return a


ST_OK, ST_RESERVED_BIT, ST_NONCANONICAL, ST_QUIRK_T0, ST_NOT_ON_CURVE, ST_NEUTRAL = range(6)

# messages of the reference's exceptions (curve4q.py:53, :62, :77 (AttributeError), :94/:448, :460)
STATUS_MESSAGES = {
    ST_RESERVED_BIT: "Malformed point: reserved bit is not zero",
    ST_NONCANONICAL: "Malformed point: reserved bit is not zero",
    ST_QUIRK_T0: "type object 'GFp' has no attribute 'two'",
    ST_NOT_ON_CURVE: "Point not on curve",
    ST_NEUTRAL: "DH computation resulted in neutral point",
}

# curve4q.py:9-20
d = (0xe40000000000000142, 0x5e472f846657e0fcb3821488f1fc0c8d)
N = 0x29cbc14e5e0a72f05397829cbc14e5dfbd004dfe0f79992fb2540ec7768ce7
Gx = (0x1A3472237C2FB305286592AD7B3833AA, 0x1E1F553F2878AA9C96869FB360AC77F6)
Gy = (0x0E3FEE9BA120785AB924A2462BCBB287, 0x6E1C4AF8630E024249A7C344844C8B5C)


def _buf(arr, shape, name):
    """Caller-provided output buffer (e.g. pinned memory from fourq_b200.pinned_empty) or a fresh array."""
    if arr is None:
        return np.empty(shape, np.uint8)
    if not isinstance(arr, np.ndarray) or arr.dtype != np.uint8 or arr.shape != tuple(shape) or not arr.flags["C_CONTIGUOUS"]:
        raise ValueError("%s must be a C-contiguous uint8 array of shape %r" % (name, tuple(shape)))
    return arr


def _raise_first(status):
    bad = np.flatnonzero(status)
    if bad.size:
        st = int(status[bad[0]])
        exc = AttributeError if st == ST_QUIRK_T0 else Exception
        raise exc("%s (row %d)" % (STATUS_MESSAGES[st], int(bad[0])))


def encode(XY, ndev=1, out=None):
    XY = _lib.rows(XY, 64, "XY")
    out = _buf(out, (XY.shape[0], 32), "out")
    _lib.check(_lib.lib().fq_encode(_lib.ptr(XY), _lib.ptr(out), XY.shape[0], ndev))
    return out


def PointOnCurve(XY, ndev=1):
    """curve4q.py:23-29 for N affine points x | y: a (N,) bool array."""
    XY = _lib.rows(XY, 64, "XY")
    ok = np.empty((XY.shape[0],), np.uint8)
    _lib.check(_lib.lib().fq_point_on_curve(_lib.ptr(XY), _lib.ptr(ok), XY.shape[0], ndev))
    return ok.astype(bool)


def decode(B, ndev=1, strict=False, out=None, status=None, spec=False):
    """decode (curve4q.py:49-96).  spec=True is an opt-in that is NOT bit-compatible with the reference on four inputs: it
    decodes as the draft specifies (t = 2 (t0 - t3) when t == 0, draft-ladd-cfrg-4q.md:865-867) where the reference raises
    AttributeError (status 3), so the encodings of (0, 1), (0, -1), (i, 0), (-i, 0) decode; everything else is unchanged."""
    B = _lib.rows(B, 32, "B")
    n = B.shape[0]
    XY = _buf(out, (n, 64), "out")
    status = _buf(status, (n,), "status")
    fn = _lib.lib().fq_decode_spec if spec else _lib.lib().fq_decode
    _lib.check(fn(_lib.ptr(B), _lib.ptr(XY), _lib.ptr(status), n, ndev))
    if strict:
        _raise_first(status)
    return XY, status


def DH(k, B, ndev=1, strict=False, out=None, status=None, algorithm=None, y_only=False):
    """encode(DH_*(k, decode(B))).  y_only=True returns the draft's shared secret instead: the y coordinate of the shared
    point as a 32-byte string (draft-ladd-cfrg-4q.md:707-714), i.e. the encoding with the sign bit of x cleared."""
    k = _lib.rows(k, 32, "k")
    B = _lib.rows(B, 32, "B")
    if k.shape[0] != B.shape[0]:
        raise ValueError("k and B must have the same number of rows")
    n = k.shape[0]
    out = _buf(out, (n, 32), "out")
    status = _buf(status, (n,), "status")
    fn = _lib.lib().fq_dh_endo if _alg(algorithm) == "endo" else _lib.lib().fq_dh
    _lib.check(fn(_lib.ptr(k), _lib.ptr(B), _lib.ptr(out), _lib.ptr(status), n, ndev))
    if y_only:
        out[:, 31] &= 0x7F
    if strict:
        _raise_first(status)
    return out, status


def DH_endo(k, XY, ndev=1, strict=False, out=None, status=None):
    return DH_windowed(k, XY, ndev=ndev, strict=strict, out=out, status=status, _fn="fq_dh_endo_affine")


def DH_windowed(k, XY, ndev=1, strict=False, out=None, status=None, _fn="fq_dh_affine"):
    k = _lib.rows(k, 32, "k")
    XY = _lib.rows(XY, 64, "XY")
    if k.shape[0] != XY.shape[0]:
        raise ValueError("k and XY must have the same number of rows")
    n = k.shape[0]
    out = _buf(out, (n, 64), "out")
    status = _buf(status, (n,), "status")
    _lib.check(getattr(_lib.lib(), _fn)(_lib.ptr(k), _lib.ptr(XY), _lib.ptr(out), _lib.ptr(status), n, ndev))
    if strict:
        _raise_first(status)
    return out, status


def DH_base(k, ndev=1, strict=False, out=None, status=None, algorithm=None):
    k = _lib.rows(k, 32, "k")
    n = k.shape[0]
    out = _buf(out, (n, 32), "out")
    status = _buf(status, (n,), "status")
    fn = getattr(_lib.lib(), {"windowed": "fq_dh_base", "endo": "fq_dh_endo_base", "comb": "fq_dh_base_comb"}[_alg(algorithm, base=True)])
    _lib.check(fn(_lib.ptr(k), _lib.ptr(out), _lib.ptr(status), n, ndev))
    if strict:
        _raise_first(status)
    return out, status


def MUL_base(k, ndev=1, out=None, algorithm=None):
    k = _lib.rows(k, 32, "k")
    out = _buf(out, (k.shape[0], 32), "out")
    fn = getattr(_lib.lib(), {"windowed": "fq_mul_base", "endo": "fq_mul_endo_base", "comb": "fq_mul_base_comb"}[_alg(algorithm, base=True)])
    _lib.check(fn(_lib.ptr(k), _lib.ptr(out), k.shape[0], ndev))
    return out


class FixedBase:
    """One public point P registered for many scalars: fixed-base DH and scalar multiplication on per-digit tables of P and
    [392]P, the comb of DH_base / MUL_base (algorithm="comb") for a point of the caller's choosing.

    P is a 32-byte encoding, or with affine=True 64-byte x | y (each half reduced mod p).  It is validated once, as DH
    validates it; an invalid P raises the reference's exception (STATUS_MESSAGES; AttributeError for the t == 0 quirk).
    Each GPU builds the tables (2 x 48,384 B) on the first call that uses them there.

    .DH(k)  per row, exactly DH(k, B) with B = P broadcast (encode(DH_windowed(k, P)) for an affine P): status 0 or 5.
    .MUL(k) per row, encode(R1toAffine(MUL_windowed(k, P))) (curve4q.py:188-235) = encode([r]P) with r = k mod N, plus N if
            that is even.  For P in the prime-order subgroup that is [k]P, and FixedBase(G).MUL(k) == MUL_base(k).  For a P
            with a small-order component it is NOT [k]P, nor what MUL_endo gives: r and k differ by a multiple of N, which
            does not annihilate the small-order part.

    close() (or the end of a `with` block, or garbage collection) frees the tables; it must not run while a call that uses
    the handle is in flight on another thread."""

    def __init__(self, P, affine=False):
        self.handle = None
        width = 64 if affine else 32
        if isinstance(P, (bytes, bytearray)):
            P = np.frombuffer(bytes(P), np.uint8)
        if not isinstance(P, np.ndarray) or P.dtype != np.uint8 or P.size != width:
            raise ValueError("P must be %d bytes (a bytes object or a uint8 array)" % width)
        P = np.ascontiguousarray(P).reshape(width)
        st = np.zeros(1, np.uint8)
        h = ctypes.c_void_p()
        _lib.check(_lib.lib().fq_base_create(_lib.ptr(P), 1 if affine else 0, _lib.ptr(st), ctypes.byref(h)))
        if st[0]:
            raise (AttributeError if st[0] == ST_QUIRK_T0 else Exception)(STATUS_MESSAGES[int(st[0])])
        self.handle = h

    def _h(self):
        if self.handle is None:
            raise ValueError("FixedBase is closed")
        return self.handle

    def DH(self, k, ndev=1, strict=False, out=None, status=None, y_only=False):
        """As DH(k, B, algorithm=any) with B = P on every row; y_only and strict as there."""
        k = _lib.rows(k, 32, "k")
        n = k.shape[0]
        out = _buf(out, (n, 32), "out")
        status = _buf(status, (n,), "status")
        _lib.check(_lib.lib().fq_dh_fixed(self._h(), _lib.ptr(k), _lib.ptr(out), _lib.ptr(status), n, ndev))
        if y_only:
            out[:, 31] &= 0x7F
        if strict:
            _raise_first(status)
        return out, status

    def MUL(self, k, ndev=1, out=None):
        k = _lib.rows(k, 32, "k")
        out = _buf(out, (k.shape[0], 32), "out")
        _lib.check(_lib.lib().fq_mul_fixed(self._h(), _lib.ptr(k), _lib.ptr(out), k.shape[0], ndev))
        return out

    def close(self):
        if self.handle is not None:
            h, self.handle = self.handle, None
            _lib.check(_lib.lib().fq_base_destroy(h))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter shutdown
            pass


def pack_affine(points):
    """[((x0, x1), (y0, y1)), ...] Python ints -> (N, 64) rows."""
    out = np.empty((len(points), 64), np.uint8)
    for i, (x, y) in enumerate(points):
        out[i] = np.frombuffer(b"".join(int(v).to_bytes(16, "little") for v in (x[0], x[1], y[0], y[1])), np.uint8)
    return out


def pack_scalars(ms):
    out = np.empty((len(ms), 32), np.uint8)
    for i, m in enumerate(ms):
        out[i] = np.frombuffer((int(m) % (1 << 256)).to_bytes(32, "little"), np.uint8)
    return out
