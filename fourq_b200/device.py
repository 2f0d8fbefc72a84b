"""Device selection, pinned host arrays and device-resident buffers (measurement helpers; bench.py uses these)."""
import ctypes

import numpy as np

from . import _lib


def device_count():
    n = _lib.lib().fq_device_count()
    if n < 0:
        _lib.check(n)
    return n


def set_device(first):
    """GPUs used by the host entry points become first .. first+ndev-1 (one process per GPU passes LOCAL_RANK)."""
    _lib.check(_lib.lib().fq_set_device_base(int(first)))


def set_select_mode(strict):
    """Table selection of every scalar multiplication: True = strict scan (default: every lane loads every table entry and
    selects in registers, no digit-dependent memory activity of any kind), False = masked loads (opt-in for non-secret
    scalars: predicated loads, no select instructions, DH 1-2 % and comb keygen 8 % faster, but the shared-memory activity of
    a load depends on how the digits are spread over a warp).  Same outputs.  FQ_STRICT_SELECT=0 selects masked loads at
    start-up."""
    _lib.check(_lib.lib().fq_set_select_mode(1 if strict else 0))


def get_select_mode():
    return bool(_lib.lib().fq_get_select_mode())


def trim():
    """Frees the per-GPU staging and scratch buffers kept between calls (they are re-allocated on demand)."""
    _lib.check(_lib.lib().fq_trim())


def last_rows_per_device(ndev):
    """Rows each of the ndev GPUs processed in the last host call of this thread (equal slices unless a GPU ran out early and helped)."""
    rows = (ctypes.c_size_t * ndev)()
    _lib.check(_lib.lib().fq_last_rows_per_device(rows, ndev))
    return [int(x) for x in rows]


def last_kernel_ms():
    return float(_lib.lib().fq_last_kernel_ms())


class _Pinned:
    def __init__(self, nbytes, rows=None, row_bytes=None, ndev=1):
        self.ptr = ctypes.c_void_p()
        if ndev > 1 and rows and _lib.lib().fq_host_alloc_sliced(ctypes.byref(self.ptr), rows, row_bytes, ndev) == _lib.FQ_OK:
            pass                      # laid out for ndev GPUs
        else:                         # one GPU, or the platform refused the placement (e.g. no host registration): ordinary page-locked memory
            self.ptr = ctypes.c_void_p()
            _lib.check(_lib.lib().fq_host_alloc(ctypes.byref(self.ptr), nbytes))
        self.nbytes = nbytes

    def __del__(self):
        try:
            if self.ptr:
                _lib.lib().fq_host_free(self.ptr)
        except Exception:  # interpreter shutdown
            pass


class _PinnedArray(np.ndarray):
    _fq_owner = None


def pinned_empty(shape, dtype=np.uint8, ndev=1):
    """numpy array backed by page-locked host memory: host entry points then copy without staging.  ndev > 1: the array is
    laid out for a call on ndev GPUs -- the bytes of GPU i's slice of rows are placed on that GPU's NUMA node
    (fq_host_alloc_sliced; an ordinary page-locked array where the platform does not allow it)."""
    shape = tuple(shape) if isinstance(shape, (tuple, list)) else (int(shape),)
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    row_bytes = (nbytes // shape[0]) if shape and shape[0] else 0
    owner = _Pinned(max(nbytes, 1), rows=shape[0] if shape else 0, row_bytes=row_bytes, ndev=ndev)
    buf = (ctypes.c_uint8 * max(nbytes, 1)).from_address(owner.ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape).view(_PinnedArray)
    arr._fq_owner = owner
    return arr


class DeviceBuffer:
    """A raw device allocation on one GPU."""

    def __init__(self, dev, nbytes):
        self.dev, self.nbytes = int(dev), int(nbytes)
        self.ptr = ctypes.c_void_p()
        _lib.check(_lib.lib().fq_dev_alloc(self.dev, ctypes.byref(self.ptr), self.nbytes))

    @classmethod
    def from_host(cls, dev, arr):
        arr = np.ascontiguousarray(arr)
        b = cls(dev, arr.nbytes)
        _lib.check(_lib.lib().fq_dev_upload(b.dev, b.ptr, _lib.ptr(arr), arr.nbytes))
        return b

    def to_host(self, shape, dtype=np.uint8):
        out = np.empty(shape, dtype)
        assert out.nbytes <= self.nbytes
        _lib.check(_lib.lib().fq_dev_download(self.dev, _lib.ptr(out), self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            _lib.check(_lib.lib().fq_dev_free(self.dev, self.ptr))
            self.ptr = ctypes.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def dev_run(op, dev, a, b, out, status, n, iters=1, c=None):
    """Launches the kernel of `op` (a key of _lib.DEVOP) on device buffers; returns average milliseconds per launch.
    c: third input operand (the condition bytes of fp_select / fp2_select)."""
    ms = ctypes.c_float()
    g = lambda x: x.ptr if x is not None else None  # noqa: E731
    _lib.check(_lib.lib().fq_dev_run3(_lib.DEVOP[op], int(dev), g(a), g(b), g(c), g(out), g(status), int(n), int(iters), ctypes.byref(ms)))
    return float(ms.value)


def dev_run_fixed(base, dh, dev, k, out, status, n, iters=1):
    """fq_dh_fixed (dh=True) or fq_mul_fixed (dh=False) of a curve4q.FixedBase on device buffers; returns average milliseconds
    per launch.  The first call on a device builds the base's tables there, before the timed launches.  status may be None
    for dh=False."""
    ms = ctypes.c_float()
    g = lambda x: x.ptr if x is not None else None  # noqa: E731
    _lib.check(_lib.lib().fq_base_dev_run(base.handle, 1 if dh else 0, int(dev), g(k), g(out), g(status), int(n), int(iters), ctypes.byref(ms)))
    return float(ms.value)


def last_phase_ms():
    """CUDA-event milliseconds of the (prepare, ladder, finish) kernels of the last launch of the last DH dev_run."""
    ms = (ctypes.c_float * 3)()
    _lib.check(_lib.lib().fq_dev_last_phase_ms(ms))
    return [float(x) for x in ms]


def flush_l2(dev):
    _lib.check(_lib.lib().fq_dev_flush_l2(int(dev)))


def imad_peak(dev=0):
    """(IMAD.WIDE.U32 per second, 32-bit IMAD per second) measured on the device: the integer-multiply roofline."""
    w, s = ctypes.c_double(), ctypes.c_double()
    _lib.check(_lib.lib().fq_imad_peak(int(dev), ctypes.byref(w), ctypes.byref(s)))
    return float(w.value), float(s.value)
