"""GPU tests of fixed-base DH and scalar multiplication for a registered point (fourq_b200.FixedBase): byte and status
equality with variable-base DH on the broadcast point, with MUL_base / DH_base for G, with the plain affine group law for
MUL on points with a small-order component, and with the C oracle on a full 2^20-row batch."""
import threading

import numpy as np
import pytest

import torsion
from oracle import c_oracle as C
from oracle import fourq_oracle as O

pytestmark = pytest.mark.gpu

# around the 256-row CTAs of k_comb and the 16-row inversion groups of k_dh_finish, several pipeline chunks, and past one chunk
SIZES = [1, 255, 256, 257, 1003, 131_083, (1 << 20) + 17]
N = O.N


@pytest.fixture(scope="module")
def fq():
    import fourq_b200
    assert fourq_b200.device_count() >= 1        # raises if the CUDA library or device is missing: no silent fallback
    return fourq_b200


@pytest.fixture(scope="module")
def kbig():
    k = np.random.default_rng(31).integers(0, 256, (SIZES[-1], 32), np.uint8)
    edge = [0, 1, 2, N - 1, N, N + 1, 2 * N, (1 << 256) - 1]
    k[:len(edge)] = np.frombuffer(b"".join(int(x % (1 << 256)).to_bytes(32, "little") for x in edge), np.uint8).reshape(-1, 32)
    return k


def _encodings(fq):
    """16 seeded prime-order points, G, 8 torsion-shifted points and 4 pure-torsion points that decode."""
    pts = [e for e, _ in torsion.prime_order_points(16, seed=41)]
    pts.append(bytes(fq.MUL_base(np.eye(1, 32, dtype=np.uint8))[0]))
    A = torsion.prime_order_points(1, seed=43)[0][1]
    tors = torsion.torsion_points()
    decodable = [T for T, o in tors if O.decode_status(torsion.enc(T))[0] == O.ST_OK]
    picks = decodable[:: max(1, len(decodable) // 8)][:8]
    pts += [torsion.enc(torsion.add(A, T)) for T in picks]
    pts += [torsion.enc(T) for T in decodable[-4:]]
    return pts


def test_dh_fixed_equals_dh_on_the_broadcast_point(fq, kbig):
    pts = _encodings(fq)
    default = fq.get_select_mode()
    try:
        for strict in (True, False):
            fq.set_select_mode(strict)
            for e in pts:
                B = np.frombuffer(e, np.uint8)
                with fq.FixedBase(e) as fb:
                    for n in SIZES:
                        k = kbig[:n]
                        want, wst = fq.DH(k, np.broadcast_to(B, (n, 32)).copy())
                        out, st = fb.DH(k)
                        assert (st == wst).all() and (out == want).all(), (e.hex(), n, strict)
    finally:
        fq.set_select_mode(default)


def test_affine_registration(fq, kbig):
    """Affine x | y, including halves written as x + p: encode(DH_windowed(k, XY))."""
    p = O.P127
    k = kbig[:1003]
    A = torsion.prime_order_points(1, seed=47)[0][1]
    T = [T for T, o in torsion.torsion_points() if o == 56][0]
    for pt in (A, torsion.add(A, T), T):
        (x0, x1), (y0, y1) = pt
        for raw in ((x0, x1, y0, y1), (x0 + p, x1, y0, y1 + p)):                  # every coordinate is below p, so x + p < 2^128
            xy = np.frombuffer(b"".join(int(v).to_bytes(16, "little") for v in raw), np.uint8)
            want, wst = fq.DH_windowed(k, np.broadcast_to(xy, (k.shape[0], 64)).copy())
            want = np.where((wst == 0)[:, None], fq.encode(want), 0)
            with fq.FixedBase(xy, affine=True) as fb:
                out, st = fb.DH(k)
            assert (st == wst).all() and (out == want).all(), raw


def test_generator_and_mul_on_torsion_shifted_points(fq, kbig):
    k = kbig[:131_083]
    G = fq.MUL_base(np.eye(1, 32, dtype=np.uint8))[0]
    with fq.FixedBase(G) as fb:
        assert (fb.MUL(k) == fq.MUL_base(k, algorithm="comb")).all()
        out, st = fb.DH(k)
        wout, wst = fq.DH_base(k)
        assert (out == wout).all() and (st == wst).all()
    A = torsion.prime_order_points(1, seed=53)[0][1]
    for o in (7, 8, 56):
        T = [T for T, oo in torsion.torsion_points() if oo == o][0]
        S = torsion.add(A, T)
        with fq.FixedBase(torsion.xy(S), affine=True) as fb:
            out = fb.MUL(k[:64])
        for i in range(0, 64, 7):
            m = int.from_bytes(bytes(k[i]), "little")
            r = m % N
            r = r + N if r % 2 == 0 else r
            assert bytes(out[i]) == torsion.enc(torsion.mul(r, S)), (o, i)


def test_invalid_points_strict_and_y_only(fq, kbig):
    e = bytearray(torsion.prime_order_points(1, seed=59)[0][0])
    bad = bytearray(e); bad[15] |= 0x80
    nonc = bytearray(32); nonc[:16] = ((1 << 127) - 1).to_bytes(16, "little")
    t0 = torsion.enc(torsion.NEUTRAL)
    for pt, st in ((bad, 1), (nonc, 2), (t0, 3)):
        assert O.decode_status(bytes(pt))[0] == st
        with pytest.raises(AttributeError if st == 3 else Exception, match=fq.STATUS_MESSAGES[st]):
            fq.FixedBase(bytes(pt))
    xy = bytearray(torsion.xy(torsion.prime_order_points(1, seed=59)[0][1])); xy[0] ^= 1
    with pytest.raises(Exception, match="Point not on curve"):
        fq.FixedBase(bytes(xy), affine=True)
    k = kbig[:1003]
    B = np.broadcast_to(np.frombuffer(bytes(e), np.uint8), (1003, 32)).copy()
    with fq.FixedBase(bytes(e)) as fb:
        assert (fb.DH(k, y_only=True)[0] == fq.DH(k, B, y_only=True)[0]).all()
        with pytest.raises(Exception, match="DH computation resulted in neutral point"):
            fb.DH(k, strict=True)                                    # k = 0, N, 2N (rows 0, 4, 6) give the neutral point
    T = [T for T, o in torsion.torsion_points() if o == 8 and O.decode_status(torsion.enc(T))[0] == 0][0]
    with fq.FixedBase(torsion.enc(T)) as fb:
        out, st = fb.DH(k)
        assert (st == 5).all() and not out.any()
    fb = fq.FixedBase(bytes(e))
    fb.close()
    with pytest.raises(ValueError):
        fb.MUL(k)


def test_threads_and_all_gpus(fq, kbig):
    n = 300_007
    k = kbig[:n]
    encs = [e for e, _ in torsion.prime_order_points(2, seed=61)]
    fbs = [fq.FixedBase(e) for e in encs]
    try:
        serial = [(fb.DH(k), fb.MUL(k)) for fb in fbs]
        errs = []

        def work(i):
            for it in range(3):
                b = (i + it) % 2
                (wo, ws), wm = serial[b]
                out, st = fbs[b].DH(k)
                if not ((out == wo).all() and (st == ws).all() and (fbs[b].MUL(k) == wm).all()):
                    errs.append((i, it))
        ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
        [t.start() for t in ts]; [t.join() for t in ts]
        assert not errs
        if fq.device_count() < 2:
            pytest.skip("one GPU: the ndev = all case needs two or more")
        nd = fq.device_count()
        for b, fb in enumerate(fbs):
            out, st = fb.DH(k, ndev=nd)
            assert (out == serial[b][0][0]).all() and (st == serial[b][0][1]).all()
            assert (fb.MUL(k, ndev=nd) == serial[b][1]).all()
    finally:
        for fb in fbs:
            fb.close()


def test_device_resident_and_a_full_batch_against_the_oracle(fq, kbig):
    from fourq_b200 import device as dev
    n = 1 << 20
    k = kbig[:n]
    e = torsion.prime_order_points(1, seed=67)[0][0]
    with fq.FixedBase(e) as fb:
        out, st = fb.DH(k)
        mo = fb.MUL(k)
        dk = dev.DeviceBuffer.from_host(0, k)
        do = dev.DeviceBuffer(0, n * 32); ds = dev.DeviceBuffer(0, n)
        assert dev.dev_run_fixed(fb, True, 0, dk, do, ds, n) > 0
        assert (do.to_host((n, 32)) == out).all() and (ds.to_host((n,)) == st).all()
        dev.dev_run_fixed(fb, False, 0, dk, do, None, n)
        assert (do.to_host((n, 32)) == mo).all()
    want, wst = C.dh(k, np.broadcast_to(np.frombuffer(e, np.uint8), (n, 32)).copy())
    assert (out == want).all() and (st == wst).all()
