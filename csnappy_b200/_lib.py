"""ctypes loader for libcsnappy_b200.so (the C-ABI boundary, include/*.h).

Fails loudly: a missing library is an ImportError-grade RuntimeError, never a
silent fallback -- there is no CPU codec in this package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CSNAPPY_B200_LIB") or os.path.join(_HERE, "libcsnappy_b200.so")  # override: kernel experiments

_lib = None

_u32p = C.POINTER(C.c_uint32)


def _declare(L):
    vp, u32, u64, i = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    sig = {
        # csnappy.h
        "csnappy_max_compressed_length": (u32, [u32]),
        "csnappy_compress_fragment": (vp, [vp, u32, vp, vp, i]),
        "csnappy_compress": (None, [vp, u32, vp, _u32p, vp, i]),
        "csnappy_get_uncompressed_length": (i, [vp, u32, _u32p]),
        "csnappy_decompress": (i, [vp, u32, vp, u32]),
        "csnappy_decompress_noheader": (i, [vp, u32, vp, _u32p]),
        # csnappy_batch.h
        "csnappy_batch_compress_fragments": (i, [vp, vp, u64, vp, u32, u32, vp, u64, vp, i, u32, vp]),
        "csnappy_batch_decompress": (i, [vp, vp, u64, vp, u32, vp, u64, vp, u32, vp, vp, u32, vp]),
        "csnappy_batch_pack": (i, [vp, u64, vp, u32, vp, vp, vp]),
        "csnappy_batch_compress_fragments_host": (i, [vp, u64, u32, u32, vp, u64, vp, i]),
        "csnappy_batch_decompress_host": (i, [vp, u64, vp, u32, vp, u64, u32, vp, vp, u32]),
        "csnappy_bc_max_container_length": (u64, [u64, u32]),
        "csnappy_bc_compress_host": (i, [vp, u64, u32, vp, u64, C.POINTER(C.c_uint64), i]),
        "csnappy_bc_decompress_host": (i, [vp, u64, u32, vp, u64, C.POINTER(C.c_uint64), _u32p]),
        "csnappy_batch_compress_workspace": (u64, [vp, u32, u32]),
        "csnappy_batch_compress": (i, [vp, vp, u64, vp, u32, u32, vp, u64, vp, i, vp, u64, vp]),
        "csnappy_bc_compress_host_multi": (i, [vp, u64, u32, vp, u64, C.POINTER(C.c_uint64), i, vp, i]),
        "csnappy_bc_decompress_host_multi": (i, [vp, u64, u32, vp, u64, C.POINTER(C.c_uint64), _u32p, vp, i]),
        "csnappy_bc_compress_workspace": (u64, [u64, u32]),
        "csnappy_bc_compress": (i, [vp, u64, u32, vp, u64, vp, i, vp, u64, vp]),
        "csnappy_bc_index": (i, [vp, u64, u32, vp, u64, _u32p, vp]),
        "csnappy_bc_decompress_pages_workspace": (u64, [u32]),
        "csnappy_bc_decompress_pages": (i, [vp, u64, u32, vp, u32, vp, u32, vp, u64, vp, vp, vp, u64, vp]),
        "csnappy_bc_decompress_workspace": (u64, [u64, u32, u64]),
        "csnappy_bc_decompress": (i, [vp, u64, u32, vp, u64, vp, vp, vp, vp, u64, vp]),
        "csnappy_stream_decompress_workspace": (u64, [u32, u32]),
        "csnappy_stream_decompress": (i, [vp, u32, vp, u32, vp, vp, vp, u64, vp]),
        "csnappy_framed_max_length": (u64, [u64]),
        "csnappy_framed_compress_workspace": (u64, [u64]),
        "csnappy_framed_compress": (i, [vp, u64, vp, u64, vp, i, vp, u64, vp]),
        "csnappy_framed_decompress_workspace": (u64, [u64]),
        "csnappy_framed_decompress": (i, [vp, u64, vp, u64, vp, vp, vp, vp, u64, vp]),
        "csnappy_framed_compress_host": (i, [vp, u64, vp, u64, C.POINTER(C.c_uint64), i]),
        "csnappy_framed_decompress_host": (i, [vp, u64, vp, u64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "csnappy_framed_crc32c": (i, [vp, u64, vp, vp]),
        "csnappy_framed_batch_compress_workspace": (u64, [vp, u32]),
        "csnappy_framed_batch_compress": (i, [vp, vp, vp, u32, vp, vp, u64, vp, i, vp, u64, vp]),
        "csnappy_framed_batch_decompress_workspace": (u64, [vp, u32]),
        "csnappy_framed_batch_decompress": (i, [vp, vp, vp, u32, vp, vp, vp, vp, vp, vp, vp, u64, vp]),
        "csnappy_framed_batch_decompressed_length": (i, [vp, vp, vp, u32, vp, vp, vp]),
        "csnappy_b200_device_count": (i, []),
        "csnappy_b200_device_ok": (i, []),
        "csnappy_b200_last_error": (C.c_char_p, []),
        "csnappy_b200_kernel_launches": (u64, []),
        "csnappy_b200_set_tuning": (i, [C.c_char_p, i]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    return sig


def lib():
    """The loaded library.  Raises if it has not been built (python -m csnappy_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m csnappy_b200.build` "
                "(nvcc + gcc; there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L._signatures = _declare(L)
        _lib = L
    return _lib


def last_error() -> str:
    return (lib().csnappy_b200_last_error() or b"").decode()
