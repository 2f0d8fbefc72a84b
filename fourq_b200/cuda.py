"""fourq_b200.cuda -- the operations on CUDA tensors, enqueued on a CUDA stream (fq_stream_run, fq_base_stream_run).

An optional adapter for PyTorch: importing this module imports torch; `import fourq_b200` does not.  Every function takes
torch.uint8 CUDA tensors of shape (N, w), C-contiguous, with the names and keywords of the numpy facade
(fourq_b200.curve4q, .curve25519, .fields), and returns tensors shaped as the facade returns arrays.

    stream   the torch.cuda.Stream to enqueue on; None = torch.cuda.current_stream() of the inputs' device.  The call returns
             at once: the results are there when the stream reaches this point, so torch work on the same stream sees them,
             and the call can be captured into a torch.cuda.CUDAGraph (after one call on that GPU outside capture).
    out, status  optional output tensors; otherwise torch.empty on the inputs' device, allocated while `stream` is current,
             so that the caching allocator ties them to that stream.  Inputs made on another stream must be ordered with
             `stream` by the caller (wait_stream / record_stream), as for any torch kernel.

There is no strict=: raising on a failed row needs the statuses on the host, which is a synchronisation.  Check the
returned status tensor where the caller is ready to wait for it.  Misuse the device cannot catch -- a CPU tensor, tensors
on two GPUs, a stream of another GPU, a misaligned view, an output that overlaps an input -- raises FourQError (or
TypeError / ValueError for dtype and shape) before anything is enqueued.
"""
import torch

from . import _lib
from .curve4q import _alg

__all__ = ["DH", "DH_windowed", "DH_endo", "DH_base", "MUL_base", "DH_fixed", "MUL_fixed", "decode", "encode", "PointOnCurve",
           "x25519", "run"]


def _rows(t, width, name, n=None):
    """Validates a (N, width) uint8 contiguous CUDA tensor, as _lib.rows does for numpy arrays."""
    if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8:
        raise TypeError("%s must be a torch.uint8 tensor of shape (N, %d)" % (name, width))
    if t.dim() != 2 or t.shape[1] != width:
        raise ValueError("%s must have shape (N, %d), got %r" % (name, width, tuple(t.shape)))
    if not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor (fourq_b200.cuda works on device memory; the numpy facade takes host arrays)" % name)
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    if n is not None and t.shape[0] != n:
        raise ValueError("%s must have %d rows, got %d" % (name, n, t.shape[0]))
    return t


def _stream(stream, t):
    return torch.cuda.current_stream(t.device) if stream is None else stream


def _buf(t, shape, name, like, stream):
    """Caller-provided output tensor, or a new one on like's device allocated under `stream`."""
    if t is None:
        with torch.cuda.stream(stream):
            return torch.empty(shape, dtype=torch.uint8, device=like.device)
    if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
        raise ValueError("%s must be a contiguous torch.uint8 tensor of shape %r" % (name, tuple(shape)))
    return t


def _p(t):
    return t.data_ptr() if t is not None else None


def _run(op, ins, out_w, status, out, st, stream):
    """fq_stream_run of `op` (a key of _lib.DEVOP) on the validated inputs; returns (out, status or None)."""
    a = ins[0]
    n = a.shape[0]
    s = _stream(stream, a)
    out = _buf(out, (n, out_w), "out", a, s)
    st = _buf(st, (n,), "status", a, s) if status else None
    ptrs = [_p(x) for x in ins] + [None] * (3 - len(ins))
    _lib.check(_lib.lib().fq_stream_run(_lib.DEVOP[op], *ptrs, _p(out), _p(st), n, s.cuda_stream))
    return out, st, s


def _y_only(out, s):
    with torch.cuda.stream(s):
        out[:, 31] &= 0x7F


def DH(k, B, out=None, status=None, algorithm=None, y_only=False, stream=None):
    """encode(DH_*(k, decode(B))) -> (out[N,32], status[N]); y_only=True clears the sign bit of x (the draft's shared secret)."""
    k = _rows(k, 32, "k")
    B = _rows(B, 32, "B", k.shape[0])
    out, st, s = _run("dh_endo" if _alg(algorithm) == "endo" else "dh", [k, B], 32, True, out, status, stream)
    if y_only:
        _y_only(out, s)
    return out, st


def DH_windowed(k, XY, out=None, status=None, stream=None, _op="dh_affine"):
    """DH_windowed(k, (x, y)) on affine rows -> (XY[N,64], status[N])."""
    k = _rows(k, 32, "k")
    XY = _rows(XY, 64, "XY", k.shape[0])
    out, st, _ = _run(_op, [k, XY], 64, True, out, status, stream)
    return out, st


def DH_endo(k, XY, out=None, status=None, stream=None):
    return DH_windowed(k, XY, out=out, status=status, stream=stream, _op="dh_endo_affine")


def DH_base(k, out=None, status=None, algorithm=None, stream=None):
    k = _rows(k, 32, "k")
    op = {"windowed": "dh_base", "endo": "dh_endo_base", "comb": "dh_base_comb"}[_alg(algorithm, base=True)]
    out, st, _ = _run(op, [k], 32, True, out, status, stream)
    return out, st


def MUL_base(k, out=None, algorithm=None, stream=None):
    k = _rows(k, 32, "k")
    op = {"windowed": "mul_base", "endo": "mul_endo_base", "comb": "mul_base_comb"}[_alg(algorithm, base=True)]
    return _run(op, [k], 32, False, out, None, stream)[0]


def DH_fixed(base, k, out=None, status=None, y_only=False, stream=None):
    """FixedBase.DH on a CUDA tensor of scalars: per row DH(k, B) with B = the registered point -> (out[N,32], status[N])."""
    k = _rows(k, 32, "k")
    n = k.shape[0]
    s = _stream(stream, k)
    out = _buf(out, (n, 32), "out", k, s)
    status = _buf(status, (n,), "status", k, s)
    _lib.check(_lib.lib().fq_base_stream_run(base._h(), 1, _p(k), _p(out), _p(status), n, s.cuda_stream))
    if y_only:
        _y_only(out, s)
    return out, status


def MUL_fixed(base, k, out=None, stream=None):
    """FixedBase.MUL on a CUDA tensor of scalars -> out[N,32]."""
    k = _rows(k, 32, "k")
    s = _stream(stream, k)
    out = _buf(out, (k.shape[0], 32), "out", k, s)
    _lib.check(_lib.lib().fq_base_stream_run(base._h(), 0, _p(k), _p(out), None, k.shape[0], s.cuda_stream))
    return out


def decode(B, out=None, status=None, spec=False, stream=None):
    """decode (curve4q.py:49-96) -> (XY[N,64], status[N]); spec=True as in fourq_b200.decode."""
    B = _rows(B, 32, "B")
    out, st, _ = _run("decode_spec" if spec else "decode", [B], 64, True, out, status, stream)
    return out, st


def encode(XY, out=None, stream=None):
    XY = _rows(XY, 64, "XY")
    return _run("encode", [XY], 32, False, out, None, stream)[0]


def PointOnCurve(XY, stream=None):
    """curve4q.py:23-29 on affine rows -> a (N,) bool tensor."""
    XY = _rows(XY, 64, "XY")
    ok = _run("on_curve", [XY], 1, False, None, None, stream)[0]
    return ok.view(torch.bool).reshape(-1)


def x25519(k, u, out=None, stream=None):
    """RFC 7748 X25519 (curve25519.py:88-91) on (N,32) rows -> out[N,32]."""
    k = _rows(k, 32, "k")
    u = _rows(u, 32, "u", k.shape[0])
    return _run("x25519", [k, u], 32, False, out, None, stream)[0]


_UNARY = ("sqr", "inv", "neg", "conj", "invsqrt")


def run(op_name, a, b=None, c=None, out=None, status=None, stream=None):
    """A field operation by its _lib.DEVOP name: fp_* on (N,16) rows, fp2_* and f25519_* on (N,32) rows; fp_select /
    fp2_select take a = x, b = y and c = the (N,) or (N,1) condition bytes.  Returns out."""
    if op_name not in _lib.DEVOP or not op_name.startswith(("fp_", "fp2_", "f25519_")):
        raise ValueError("run() takes the field operations of _lib.DEVOP (fp_*, fp2_*, f25519_*); the curve operations have their own functions")
    if status is not None:
        raise ValueError("the field operations have no status")
    w = 16 if op_name.startswith("fp_") else 32
    a = _rows(a, w, "a")
    ins = [a]
    if op_name.endswith("select"):
        if c is None or not isinstance(c, torch.Tensor):
            raise TypeError("c must be a torch.uint8 tensor of condition bytes")
        ins += [_rows(b, w, "b", a.shape[0]), _rows(c.reshape(-1, 1) if c.dim() == 1 else c, 1, "c", a.shape[0])]
    elif op_name.split("_", 1)[1] not in _UNARY:
        ins.append(_rows(b, w, "b", a.shape[0]))
    return _run(op_name, ins, w, False, out, None, stream)[0]
