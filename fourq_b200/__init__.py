"""fourq_b200 -- B200-native batched Curve4Q (FourQ).

Drop-in, batched counterparts of the reference's Python entry points (bifurcation/fourq impl/curve4q.py, fields.py,
curve25519.py): every argument and result is a C-contiguous numpy uint8 array with one 32-byte (or 64-byte affine)
row per element.  All arithmetic runs in hand-written CUDA kernels for sm_100a behind a C ABI
(include/fourq_b200.h, libfourq_b200.so, loaded with ctypes); there is no CPU implementation.
"""
from ._lib import FourQError, lib  # noqa: F401
from . import curve4q, fields, curve25519, device  # noqa: F401
from .curve4q import (decode, encode, DH, DH_windowed, DH_endo, DH_base, MUL_base, FixedBase, STATUS_MESSAGES,  # noqa: F401
                      ST_OK, ST_RESERVED_BIT, ST_NONCANONICAL, ST_QUIRK_T0, ST_NOT_ON_CURVE, ST_NEUTRAL)
from .fields import GFp, GFp2, GFp25519  # noqa: F401
from .curve25519 import x25519  # noqa: F401
from .device import set_device, device_count, pinned_empty, last_kernel_ms, set_select_mode, get_select_mode, trim  # noqa: F401

__all__ = ["decode", "encode", "DH", "DH_windowed", "DH_endo", "DH_base", "MUL_base", "FixedBase", "GFp", "GFp2", "GFp25519", "x25519", "set_device",
           "device_count", "pinned_empty", "last_kernel_ms", "set_select_mode", "get_select_mode", "trim", "FourQError"]
