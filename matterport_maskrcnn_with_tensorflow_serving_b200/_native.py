"""ctypes binding of lib/libmrx.so (C ABI: include/mrx.h).

There is no CPU fallback: if the library is missing or a call fails, this raises.
PyTorch is imported first so that libmrx.so resolves libcudart.so.12 to the CUDA
runtime instance torch already loaded (shared device / stream state).
"""
from __future__ import annotations

import ctypes as C
import os
import re

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# MRX_LIB=<file name under lib/> selects another build of the library (development only:
# e.g. libmrx_dev.so built with MRX_NVCC_FLAGS=-DMRX_DEV); the default is the shipped one
LIB_PATH = os.path.join(_PKG_DIR, "lib", os.environ.get("MRX_LIB", "libmrx.so"))
HEADER_PATH = os.path.join(os.path.dirname(_PKG_DIR), "include", "mrx.h")

MRX_OK = 0
MRX_F32 = 0
MRX_F64 = 1
MRX_ST_CLASS_RANGE = 1
MRX_ST_BOX_RANGE = 2
MRX_GEOM_INTS = 8
MRX_MAX_BATCH = 4096
ABI_VERSION = 6
MRX_SCHED_WORDS = 4
MRX_PEER_HANDLE_BYTES = 64


class MrxError(RuntimeError):
    """A libmrx call returned a negative status."""


_vp, _i, _ip = C.c_void_p, C.c_int, C.POINTER(C.c_int)
_dp = C.POINTER(C.c_double)

# name -> (restype, argtypes); must list every function include/mrx.h declares
SIGNATURES = {
    "mrx_abi_version": (_i, []),
    "mrx_last_error": (C.c_char_p, []),
    "mrx_device_props": (_i, [_i, _ip, _ip, _ip, _ip]),
    "mrx_anchor_count": (_i, [_i, _i, _ip, _i, _i, _i, C.POINTER(C.c_longlong)]),
    "mrx_anchors": (_i, [_vp, _i, _i, _dp, _dp, _ip, _i, _i, _i, _vp]),
    "mrx_unmold_prologue": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _vp]),
    "mrx_gather_tiles": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "mrx_unmold_prepare": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp,
                                _vp, _vp, _vp, _vp, _vp]),
    "mrx_mask_expand": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp,
                             _vp]),
    "mrx_mask_expand_values": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i,
                                    _vp, _vp]),
    "mrx_mask_expand_packed": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp,
                                    _vp]),
    "mrx_rle_count": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "mrx_rle_write": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "mrx_contours_count": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "mrx_contours_write": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                C.c_longlong, _i, _i, _i, _i, _vp]),
    "mrx_peer_alloc": (_i, [C.c_ulonglong, C.POINTER(C.c_void_p)]),
    "mrx_peer_free": (_i, [_vp]),
    "mrx_peer_export": (_i, [_vp, C.c_char_p]),
    "mrx_peer_open": (_i, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "mrx_peer_close": (_i, [_vp]),
    "mrx_peer_signal": (_i, [_vp, C.c_uint, _vp]),
    "mrx_peer_wait": (_i, [_vp, _i, C.c_uint, _vp]),
    "mrx_cv2_resize_u8c3": (_i, [_vp, _i, _i, _vp, _i, _i, _vp]),
    "mrx_mold_image": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _dp, _i, _vp, _vp, _vp]),
    "mrx_cv2_resize_u8c3_batch": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "mrx_mold_image_batch": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _dp, _i, _vp, _vp,
                                  _vp]),
    "mrx_composite_masks": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_double, _vp, _i, _i,
                                 C.c_longlong, _vp]),
    "mrx_pack_masks": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
}

_lib = None


def declared_symbols(header_path=HEADER_PATH):
    """Function names declared in include/mrx.h (used by the symbol-export test)."""
    with open(header_path) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mrx_[a-z0-9_]+)\s*\(", text)))


def load(build_if_missing=True):
    """Load libmrx.so (building it in-tree first if it is absent). Raises on failure."""
    global _lib
    if _lib is not None:
        return _lib
    import torch  # noqa: F401  (loads libcudart.so.12 before libmrx.so asks for it)

    default_lib = os.path.basename(LIB_PATH) == "libmrx.so"
    if build_if_missing and default_lib:
        # cheap when nothing changed (a digest of the sources against lib/libmrx.stamp); a stale
        # library whose ABI number happens to match is rebuilt instead of silently used.  Without
        # nvcc (a deployment box) the prebuilt library is used as it is.
        from . import build as _build
        try:
            _build.build()
        except RuntimeError:
            if not os.path.exists(LIB_PATH):
                raise
    if not os.path.exists(LIB_PATH):
        raise MrxError(f"{LIB_PATH} is missing; run __graft_entry__.build()")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    got = lib.mrx_abi_version()
    if got != ABI_VERSION:
        raise MrxError(f"libmrx ABI {got} != expected {ABI_VERSION}; rebuild the library")
    _lib = lib
    return lib


def check(rc, what):
    if rc != MRX_OK:
        msg = load().mrx_last_error()
        raise MrxError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")


def int_array(values):
    arr = (C.c_int * len(values))(*[int(v) for v in values])
    return arr


def double_array(values):
    arr = (C.c_double * len(values))(*[float(v) for v in values])
    return arr


def stream_ptr(stream):
    """cudaStream_t of a torch.cuda.Stream (or the current stream) as an integer."""
    import torch

    if stream is None:
        stream = torch.cuda.current_stream()
    return C.c_void_p(stream.cuda_stream)


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise MrxError("no CUDA device: this package has no CPU fallback "
                       "(the CPU restatement under oracle/ is test infrastructure only)")
