"""GPU tests on points with a small-order component (tests/torsion.py), the input a small-subgroup attack sends to
variable-base DH: the 392 points of the 392-torsion subgroup and prime-order points shifted by them.  DH_core clears the
cofactor before the ladder, so a pure torsion point gives the neutral point (status 5, or 3 where decode stops at the
reference's t == 0 quirk) and DH(k, P + T) == DH(k, P).  For the kernels these are exceptional rows: the endomorphisms and
the table run on the neutral point, and k_dh_finish inverts neutral rows in the same 16-row groups as good ones.  Every row
is compared with the C oracle; at size the shift property is checked without one."""
import numpy as np
import pytest

import torsion
from oracle import c_oracle as C
from oracle import fourq_oracle as O

pytestmark = pytest.mark.gpu

# ragged batch sizes: inside and across the 16-row inversion groups of k_dh_finish and the 128-row CTAs of k_dh_prep
SIZES = [1, 15, 16, 17, 1003, 131_083]


@pytest.fixture(scope="module")
def fq():
    import fourq_b200
    assert fourq_b200.device_count() >= 1        # raises if the CUDA library or device is missing: no silent fallback
    return fourq_b200


@pytest.fixture(scope="module")
def tgrid():
    k, enc, same = torsion.grid()
    want, wst = C.dh(k, enc)
    return k, enc, same, want, wst


@pytest.fixture(scope="module")
def tagrid():
    k, xy, same = torsion.affine_grid()
    want, wst = C.dh_affine(k, xy)
    return k, xy, same, want, wst


def _check_grid_shape(same, out, st):
    """What the oracle comparison already implies, stated on its own: torsion rows are failures with zero-filled rows, and
    every shifted row equals its unshifted row."""
    tors = same < 0
    assert set(np.unique(st[tors])) <= {3, 5} and not out[tors].any()
    assert not st[~tors].any() and (out[~tors] == out[same[~tors]]).all()


@pytest.mark.parametrize("alg", ["endo", "windowed"])
def test_torsion_grid_both_select_modes(fq, tgrid, tagrid, alg):
    """fq.DH and the affine entry point of one algorithm on the torsion grids, strict scan and masked loads, against the C oracle."""
    k, enc, same, want, wst = tgrid
    ka, xy, samea, wanta, wsta = tagrid
    aff = fq.DH_endo if alg == "endo" else fq.DH_windowed
    default = fq.get_select_mode()
    try:
        for strict in (True, False):
            fq.set_select_mode(strict)
            out, st = fq.DH(k, enc, algorithm=alg)
            assert (st == wst).all() and (out == want).all(), strict
            _check_grid_shape(same, out, st)
            out, st = aff(ka, xy)
            assert (st == wsta).all() and (out == wanta).all(), strict
            _check_grid_shape(samea, out, st)
            assert (st[samea < 0] == 5).all()                     # the affine path reaches DH_core on the order-1, 2, 4 points too
    finally:
        fq.set_select_mode(default)


def _mixed_batch(fq, n, grid_pt, affine, seed):
    """n rows: random scalars against prime-order points, with grid rows (all of them, or n // 2 at random for small n) at
    random positions.  Returns (k, points)."""
    gk, gp = grid_pt
    rng = np.random.default_rng(seed)
    k = rng.integers(0, 256, (n, 32), np.uint8)
    pub = fq.MUL_base(rng.integers(0, 256, (n, 32), np.uint8))
    pt = C.decode(pub)[0] if affine else pub
    m = min(len(gk), max(1, n // 2))
    src = rng.choice(len(gk), m, replace=False)
    dst = rng.choice(n, m, replace=False)
    k[dst] = gk[src]; pt[dst] = gp[src]
    return k, pt


@pytest.mark.parametrize("n", SIZES)
def test_torsion_rows_in_ragged_batches(fq, tgrid, tagrid, n):
    """Torsion and shifted rows shuffled into batches of good rows, so that neutral results share inversion groups and CTAs
    with good rows; both algorithms, encoded and affine entry points, every row against the C oracle."""
    k, pub = _mixed_batch(fq, n, tgrid[:2], False, n)
    want, wst = C.dh(k, pub)
    if n >= 16:
        assert (wst == 5).any() and (wst == 0).any()
    for alg in ("endo", "windowed"):
        out, st = fq.DH(k, pub, algorithm=alg)
        assert (st == wst).all() and (out == want).all(), alg
    k, xy = _mixed_batch(fq, n, tagrid[:2], True, n + 1)
    want, wst = C.dh_affine(k, xy)
    for fn in (fq.DH_endo, fq.DH_windowed):
        out, st = fn(k, xy)
        assert (st == wst).all() and (out == want).all(), fn.__name__


def test_decode_and_on_curve_on_torsion_points(fq, tgrid):
    """decode, decode(spec=True) and PointOnCurve on the encodings and x | y rows of all 392 torsion points (and the shifted
    points of the grid), against the oracle: the reference's decode stops at the t == 0 quirk on exactly the points of order
    1, 2 and 4; the draft's decode recovers every point."""
    tors = torsion.torsion_points()
    enc = np.array([np.frombuffer(torsion.enc(T), np.uint8) for T, _ in tors])
    xy = np.array([np.frombuffer(torsion.xy(T), np.uint8) for T, _ in tors])
    small = np.array([o <= 4 for _, o in tors])
    assert small.sum() == 4
    got, st = fq.decode(enc)
    want, wst = C.decode(enc)
    assert (st == wst).all() and (got == want).all()
    assert (st[small] == 3).all() and not st[~small].any() and (got[~small] == xy[~small]).all()
    got, st = fq.decode(enc, spec=True)
    assert [(bytes(a), int(b)) for a, b in zip(got, st)] == [O.row_decode(bytes(e), spec=True) for e in enc]
    assert not st.any() and (got == xy).all()
    assert fq.curve4q.PointOnCurve(xy).all() and (C.on_curve(xy)).all()
    bad = xy.copy(); bad[:, 40] ^= 1                                           # y0 off by a bit: off the curve
    assert not fq.curve4q.PointOnCurve(bad).any() and not C.on_curve(bad).any()
    genc = tgrid[1]
    got, st = fq.decode(genc)
    want, wst = C.decode(genc)
    assert (st == wst).all() and (got == want).all()
    assert (fq.curve4q.PointOnCurve(got[st == 0])).all()


def test_dh_torsion_shift_property_at_size(fq):
    """DH(k, P + T) == DH(k, P) on 2^18 rows: 4,096 prime-order points from fq.MUL_base, each shifted by the 64 torsion points
    of one fixed subset (the 8 points of order dividing 8 and 56 others), a fresh scalar per row; both algorithms.  No oracle
    needed: P + T is built with the plain group law of tests/torsion.py."""
    rng = np.random.default_rng(392)
    tors = torsion.torsion_points()
    pick = [i for i, (_, o) in enumerate(tors) if 8 % o == 0]
    rest = [i for i in range(len(tors)) if i not in pick]
    pick += sorted(rng.choice(rest, 64 - len(pick), replace=False).tolist())
    Ts = [tors[i][0] for i in pick]
    npts = 4096
    pub = fq.MUL_base(rng.integers(0, 256, (npts, 32), np.uint8))
    xy, st = fq.decode(pub)
    assert not st.any()
    Ps = [O.xy_from_bytes(bytes(r)) for r in xy]
    shifted = np.frombuffer(b"".join(torsion.shifted(A, T)[1] for A in Ps for T in Ts), np.uint8).reshape(-1, 32)
    n = npts * len(Ts)
    assert n == 1 << 18
    k = rng.integers(0, 256, (n, 32), np.uint8)
    unshifted = np.repeat(pub, len(Ts), axis=0)
    for alg in ("endo", "windowed"):
        a, sa = fq.DH(k, shifted, algorithm=alg)
        b, sb = fq.DH(k, unshifted, algorithm=alg)
        assert not sa.any() and not sb.any(), alg
        assert (a == b).all(), alg
    want, wst = C.dh(k[::61], shifted[::61])
    assert not wst.any() and (want == a[::61]).all()


def test_device_resident_path_on_torsion_grid(fq, tgrid, tagrid):
    """fq_dev_run (the path the benchmark measures) with dh, dh_endo, dh_affine and dh_endo_affine on the torsion grids: the same
    bytes as the host path and the oracle."""
    for op, alg, (k, pt, same, want, wst) in (("dh", "windowed", tgrid), ("dh_endo", "endo", tgrid),
                                               ("dh_affine", "windowed", tagrid), ("dh_endo_affine", "endo", tagrid)):
        n, w = len(k), pt.shape[1]
        dk = fq.device.DeviceBuffer.from_host(0, k); dp = fq.device.DeviceBuffer.from_host(0, pt)
        do = fq.device.DeviceBuffer(0, n * w); ds = fq.device.DeviceBuffer(0, n)
        fq.device.dev_run(op, 0, dk, dp, do, ds, n)
        got, st = do.to_host((n, w)), ds.to_host((n,))
        if w == 32:
            host, hst = fq.DH(k, pt, algorithm=alg)
        else:
            host, hst = (fq.DH_endo if alg == "endo" else fq.DH_windowed)(k, pt)
        assert (got == host).all() and (st == hst).all(), op
        assert (got == want).all() and (st == wst).all(), op
        for b in (dk, dp, do, ds):
            b.free()
