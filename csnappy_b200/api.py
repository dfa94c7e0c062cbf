"""Python mirror of the reference's C interface, bound to libcsnappy_b200.so.

Names, argument meaning and error behaviour follow /root/reference/csnappy.h:30-129
so that the parity tests read like the reference's own callers (cl_tester.c:14-114,
167-238; block_compressor.c:113-134).  Every function below goes through the C-ABI
(ctypes) into the CUDA kernels; nothing here compresses or decompresses on the CPU.

Host-buffer calls (bytes in / bytes out):
    csnappy_max_compressed_length, csnappy_compress_fragment, csnappy_compress,
    csnappy_get_uncompressed_length, csnappy_decompress, csnappy_decompress_noheader
Device-resident batches (torch CUDA tensors, asynchronous on the current stream):
    batch_compress_fragments, batch_decompress, batch_pack
Host-buffer batches (numpy / pinned torch tensors, synchronous, pipelined H2D/D2H):
    batch_compress_fragments_host, batch_decompress_host
block_compressor page container: bc_compress_host, bc_decompress_host (host buffers); bc_compress_device,
    bc_index_device, bc_decompress_pages_device (random page reads), bc_decompress_device (CUDA tensors, current
    stream)
Snappy framing format (64 KiB chunks with masked CRC-32C):
    framed_compress, framed_decompress (host bytes); framed_compress_device, framed_decompress_device,
    framed_crc32c_device (CUDA tensors, current stream); many streams in one call: framed_batch_compress,
    framed_batch_decompress (lists of bytes) and framed_batch_compress_device, framed_batch_decompress_device,
    framed_batch_decompressed_length_device (CUDA tensors, host offset / length arrays)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._lib import last_error, lib

CSNAPPY_VERSION = 5
CSNAPPY_WORKMEM_BYTES_POWER_OF_TWO = 16
CSNAPPY_WORKMEM_BYTES = 1 << 16
CSNAPPY_E_OK = 0
CSNAPPY_E_HEADER_BAD = -1
CSNAPPY_E_OUTPUT_INSUF = -2
CSNAPPY_E_OUTPUT_OVERRUN = -3
CSNAPPY_E_INPUT_NOT_CONSUMED = -4
CSNAPPY_E_DATA_MALFORMED = -5
CSNAPPY_E_DEVICE = -100
CSNAPPY_E_BAD_ARG = -101
BATCH_SHRINK_TABLE = 1
BATCH_WITH_HEADER = 2
BATCH_RAW_IF_FULL = 4
FRAGMENT_MAX = 32768


class CsnappyDeviceError(RuntimeError):
    pass


def _check(rc: int, what: str):
    if rc != 0:
        raise CsnappyDeviceError(f"{what} failed (rc={rc}): {last_error()}")


def _in_buf(data) -> np.ndarray:
    a = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    if a.size == 0:
        a = np.zeros(1, dtype=np.uint8)
    return np.ascontiguousarray(a)


# ----------------------------------------------------------------------------- csnappy.h mirror
def csnappy_max_compressed_length(source_len: int) -> int:
    return lib().csnappy_max_compressed_length(source_len)


def csnappy_compress_fragment(data: bytes, workmem_bytes_power_of_two: int = 15) -> bytes:
    """One fragment (<= 32 KiB), no length prefix.  csnappy.h:46-52."""
    n = len(data)
    src = _in_buf(data)
    out = np.empty(csnappy_max_compressed_length(n), dtype=np.uint8)
    end = lib().csnappy_compress_fragment(src.ctypes.data, n, out.ctypes.data, None, workmem_bytes_power_of_two)
    return out[: end - out.ctypes.data].tobytes()


def csnappy_compress(data: bytes, workmem_bytes_power_of_two: int = CSNAPPY_WORKMEM_BYTES_POWER_OF_TWO) -> bytes:
    """Whole buffer with varint32 prefix.  csnappy.h:65-72."""
    n = len(data)
    src = _in_buf(data)
    out = np.empty(csnappy_max_compressed_length(n) + 32 * (n // FRAGMENT_MAX + 1), dtype=np.uint8)
    olen = C.c_uint32(0)
    lib().csnappy_compress(src.ctypes.data, n, out.ctypes.data, C.byref(olen), None, workmem_bytes_power_of_two)
    return out[: olen.value].tobytes()


def csnappy_get_uncompressed_length(data: bytes):
    """-> (rc, value): rc = header bytes consumed (1..5) or CSNAPPY_E_HEADER_BAD.  csnappy.h:83-87."""
    src = _in_buf(data)
    val = C.c_uint32(0)
    rc = lib().csnappy_get_uncompressed_length(src.ctypes.data, len(data), C.byref(val))
    return rc, val.value


def csnappy_decompress(data: bytes, dst_len: int):
    """-> (rc, dst bytes[0:dst_len]).  csnappy.h:99-104."""
    src = _in_buf(data)
    out = np.zeros(max(dst_len, 1), dtype=np.uint8)
    rc = lib().csnappy_decompress(src.ctypes.data, len(data), out.ctypes.data, dst_len)
    return rc, out[:dst_len].tobytes()


def csnappy_decompress_noheader(data: bytes, dst_capacity: int):
    """-> (rc, produced bytes or None).  *dst_len is only meaningful on success.  csnappy.h:114-119."""
    src = _in_buf(data)
    out = np.zeros(max(dst_capacity, 1), dtype=np.uint8)
    dl = C.c_uint32(dst_capacity)
    rc = lib().csnappy_decompress_noheader(src.ctypes.data, len(data), out.ctypes.data, C.byref(dl))
    if rc != 0:
        assert dl.value == dst_capacity, "*dst_len must be untouched on error"
        return rc, None
    return rc, out[: dl.value].tobytes()


# ----------------------------------------------------------------------------- device batches
def _stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def out_stride_for(block_len: int) -> int:
    """Output slot stride for compression: max_compressed_length rounded up to 16 bytes."""
    return (32 + block_len + block_len // 6 + 15) // 16 * 16


def batch_compress_fragments(d_in, block_len: int, n_blocks: int, wm: int, *, in_stride: int | None = None,
                             in_len=None, in_off=None, out=None, out_len=None, out_stride: int | None = None,
                             flags: int = 0):
    """Device-resident batch of csnappy_compress_fragment.  d_in: uint8 CUDA tensor.
    Returns (out uint8 [n_blocks*out_stride], out_len int32-as-uint32 [n_blocks]) CUDA tensors."""
    import torch

    in_stride = block_len if in_stride is None else in_stride
    out_stride = out_stride_for(block_len) if out_stride is None else out_stride
    if out is None:
        out = torch.empty(max(n_blocks * out_stride, 16), dtype=torch.uint8, device=d_in.device)
    if out_len is None:
        out_len = torch.empty(max(n_blocks, 1), dtype=torch.int32, device=d_in.device)
    rc = lib().csnappy_batch_compress_fragments(_ptr(d_in), _ptr(in_off), in_stride, _ptr(in_len), block_len,
                                                 n_blocks, _ptr(out), out_stride, _ptr(out_len), wm, flags,
                                                 _stream_ptr())
    _check(rc, "csnappy_batch_compress_fragments")
    return out, out_len


def batch_decompress(d_in, in_len, n_blocks: int, out_cap: int, *, in_stride: int = 0, in_off=None, out=None,
                     out_stride: int | None = None, out_caps=None, out_len=None, status=None, flags: int = 0):
    """Device-resident batch of csnappy_decompress_noheader (or csnappy_decompress with BATCH_WITH_HEADER).
    Returns (out, out_len, status) CUDA tensors."""
    import torch

    out_stride = (out_cap + 15) // 16 * 16 if out_stride is None else out_stride
    if out is None:
        out = torch.empty(max(n_blocks * out_stride, 16), dtype=torch.uint8, device=d_in.device)
    if out_len is None:
        out_len = torch.empty(max(n_blocks, 1), dtype=torch.int32, device=d_in.device)
    if status is None:
        status = torch.empty(max(n_blocks, 1), dtype=torch.int32, device=d_in.device)
    rc = lib().csnappy_batch_decompress(_ptr(d_in), _ptr(in_off), in_stride, _ptr(in_len), n_blocks, _ptr(out),
                                         out_stride, _ptr(out_caps), out_cap, _ptr(out_len), _ptr(status), flags,
                                         _stream_ptr())
    _check(rc, "csnappy_batch_decompress")
    return out, out_len, status


def batch_pack(d_slots, slot_stride: int, d_len, n_blocks: int, packed=None):
    """Exclusive scan of sizes + gather of slots.  Returns (packed uint8, off int64 [n_blocks+1])."""
    import torch

    off = torch.empty(n_blocks + 1, dtype=torch.int64, device=d_slots.device)
    if packed is None:
        packed = torch.empty(max(n_blocks * slot_stride, 16), dtype=torch.uint8, device=d_slots.device)
    rc = lib().csnappy_batch_pack(_ptr(d_slots), slot_stride, _ptr(d_len), n_blocks, _ptr(packed), _ptr(off),
                                   _stream_ptr())
    _check(rc, "csnappy_batch_pack")
    return packed, off


# ----------------------------------------------------------------------------- host batches
def _host_ptr(x):
    return x.ctypes.data if isinstance(x, np.ndarray) else x.data_ptr()


def batch_compress_fragments_host(h_in, block_len: int, n_blocks: int, wm: int, h_out, h_out_len, *,
                                  in_stride: int | None = None, out_stride: int | None = None):
    """Host buffers (numpy arrays or pinned torch CPU tensors); synchronous."""
    in_stride = block_len if in_stride is None else in_stride
    out_stride = out_stride_for(block_len) if out_stride is None else out_stride
    rc = lib().csnappy_batch_compress_fragments_host(_host_ptr(h_in), in_stride, block_len, n_blocks,
                                                      _host_ptr(h_out), out_stride, _host_ptr(h_out_len), wm)
    _check(rc, "csnappy_batch_compress_fragments_host")


def batch_decompress_host(h_in, in_stride: int, h_in_len, n_blocks: int, h_out, out_stride: int, out_cap: int,
                          h_out_len, h_status, flags: int = 0):
    rc = lib().csnappy_batch_decompress_host(_host_ptr(h_in), in_stride, _host_ptr(h_in_len), n_blocks,
                                              _host_ptr(h_out), out_stride, out_cap, _host_ptr(h_out_len),
                                              _host_ptr(h_status), flags)
    _check(rc, "csnappy_batch_decompress_host")


# ----------------------------------------------------------------------------- block_compressor container
def bc_max_container_length(input_length: int, page_size: int = 4096) -> int:
    return lib().csnappy_bc_max_container_length(input_length, page_size)


def bc_compress_host(h_in, input_length: int, h_container, wm: int = 13, page_size: int = 4096) -> int:
    """block_compressor-style container of `input_length` bytes at h_in (numpy / pinned torch) into
    h_container; returns the container length.  Reference: block_compressor.c:275-345."""
    clen = C.c_uint64(0)
    cap = h_container.nbytes if isinstance(h_container, np.ndarray) else h_container.numel() * h_container.element_size()
    rc = lib().csnappy_bc_compress_host(_host_ptr(h_in), input_length, page_size, _host_ptr(h_container), cap,
                                        C.byref(clen), wm)
    _check(rc, "csnappy_bc_compress_host")
    return clen.value


def bc_decompress_host(h_container, container_length: int, h_out, page_size: int = 4096):
    """-> (rc, bytes produced, failed page or None).  Reference: block_compressor.c:347-394."""
    olen = C.c_uint64(0)
    bad = C.c_uint32(0xFFFFFFFF)
    cap = h_out.nbytes if isinstance(h_out, np.ndarray) else h_out.numel() * h_out.element_size()
    rc = lib().csnappy_bc_decompress_host(_host_ptr(h_container), container_length, page_size, _host_ptr(h_out), cap,
                                          C.byref(olen), C.byref(bad))
    if rc in (CSNAPPY_E_DEVICE, CSNAPPY_E_BAD_ARG):
        _check(rc, "csnappy_bc_decompress_host")
    return rc, olen.value, (bad.value if rc != 0 and bad.value != 0xFFFFFFFF else None)


def bc_compress_host_multi(h_in, input_length: int, h_container, wm: int = 13, page_size: int = 4096, devices=None) -> int:
    """bc_compress_host over several devices from this one process (devices: list of device indices, None = all
    visible).  Same bytes as the single-device call."""
    clen = C.c_uint64(0)
    cap = h_container.nbytes if isinstance(h_container, np.ndarray) else h_container.numel() * h_container.element_size()
    dev = (C.c_int * len(devices))(*devices) if devices else None
    rc = lib().csnappy_bc_compress_host_multi(_host_ptr(h_in), input_length, page_size, _host_ptr(h_container), cap,
                                              C.byref(clen), wm, dev, len(devices) if devices else 0)
    _check(rc, "csnappy_bc_compress_host_multi")
    return clen.value


def bc_decompress_host_multi(h_container, container_length: int, h_out, page_size: int = 4096, devices=None):
    """-> (rc, bytes produced, failed page or None) over several devices."""
    olen = C.c_uint64(0)
    bad = C.c_uint32(0xFFFFFFFF)
    cap = h_out.nbytes if isinstance(h_out, np.ndarray) else h_out.numel() * h_out.element_size()
    dev = (C.c_int * len(devices))(*devices) if devices else None
    rc = lib().csnappy_bc_decompress_host_multi(_host_ptr(h_container), container_length, page_size, _host_ptr(h_out),
                                                cap, C.byref(olen), C.byref(bad), dev, len(devices) if devices else 0)
    if rc in (CSNAPPY_E_DEVICE, CSNAPPY_E_BAD_ARG):
        _check(rc, "csnappy_bc_decompress_host_multi")
    return rc, olen.value, (bad.value if rc != 0 and bad.value != 0xFFFFFFFF else None)


BC_NO_PAGE = 2**64 - 1  # index entry of a page outside the decodable prefix (read as -1 from an int64 tensor)


def _ws(nbytes: int, device):
    """A workspace tensor; a workspace function's UINT64_MAX (arguments beyond the limits) is left to the C call to
    refuse."""
    import torch

    return torch.empty(max(nbytes, 1) if nbytes < 1 << 62 else 1, dtype=torch.uint8, device=device)


def bc_compress_device(d_in, input_length: int | None = None, wm: int = 13, page_size: int = 4096, *, out=None,
                       out_length=None, workspace=None):
    """Page container of a uint8 CUDA tensor written on the device, asynchronous on the current stream; the same bytes
    as bc_compress_host.  Returns (container uint8 [bc_max_container_length(n)], length int64 [1]) CUDA tensors."""
    import torch

    n = d_in.numel() if input_length is None else input_length
    if out is None:
        out = torch.empty(max(bc_max_container_length(n, page_size), 1), dtype=torch.uint8, device=d_in.device)
    if out_length is None:
        out_length = torch.empty(1, dtype=torch.int64, device=d_in.device)
    if workspace is None:
        workspace = _ws(lib().csnappy_bc_compress_workspace(n, page_size), d_in.device)
    rc = lib().csnappy_bc_compress(_ptr(d_in), n, page_size, _ptr(out), out.numel(), _ptr(out_length), wm,
                                   _ptr(workspace), workspace.numel(), _stream_ptr())
    _check(rc, "csnappy_bc_compress")
    return out, out_length  # the workspace is freed in stream order, as in framed_compress_device


def bc_index_device(d_container, container_length: int | None = None, page_size: int = 4096, *, index=None):
    """Payload offset of every page of a container in device memory (the call reads the page count back).
    Returns (rc, index int64 CUDA tensor, nr_pages): rc 0, or CSNAPPY_E_DATA_MALFORMED for a container shorter than
    its index.  index[i] is -1 (BC_NO_PAGE) from the first malformed entry on.  Without `index`, one is allocated for
    the page count (a first call reads the count)."""
    import torch

    n = d_container.numel() if container_length is None else container_length
    nr = C.c_uint32(0)
    if index is None:
        rc = lib().csnappy_bc_index(_ptr(d_container), n, page_size, None, 0, C.byref(nr), _stream_ptr())
        if rc == CSNAPPY_E_BAD_ARG and nr.value:  # the count was read: size the index and ask again
            rc = 0
        if rc == CSNAPPY_E_DATA_MALFORMED:
            return rc, torch.empty(0, dtype=torch.int64, device=d_container.device), nr.value
        _check(rc, "csnappy_bc_index")
        index = torch.empty(max(nr.value, 1), dtype=torch.int64, device=d_container.device)
    rc = lib().csnappy_bc_index(_ptr(d_container), n, page_size, _ptr(index), index.numel(), C.byref(nr), _stream_ptr())
    if rc != CSNAPPY_E_DATA_MALFORMED:
        _check(rc, "csnappy_bc_index")
    return rc, index, nr.value


def bc_decompress_pages_device(d_container, index, nr_pages: int, pages, page_size: int = 4096,
                               container_length: int | None = None, *, out=None, out_stride: int | None = None,
                               out_len=None, status=None, workspace=None):
    """Decode the pages numbered by `pages` (int32 CUDA tensor, read as uint32) of a container in device memory, with
    `index` / `nr_pages` from bc_index_device; request k goes to out[k * out_stride, + page_size).  Asynchronous on
    the current stream.  Returns (out uint8, out_len int32, status int32) CUDA tensors; status per request: 0, the
    page's decode result, CSNAPPY_E_DATA_MALFORMED (page outside the decodable prefix) or CSNAPPY_E_BAD_ARG (page
    number >= nr_pages)."""
    import torch

    n = pages.numel()
    size = d_container.numel() if container_length is None else container_length
    out_stride = page_size if out_stride is None else out_stride
    dev = d_container.device
    if out is None:
        out = torch.empty(max(n * out_stride, 1), dtype=torch.uint8, device=dev)
    if out_len is None:
        out_len = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    if status is None:
        status = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    if workspace is None:
        workspace = _ws(lib().csnappy_bc_decompress_pages_workspace(n), dev)
    rc = lib().csnappy_bc_decompress_pages(_ptr(d_container), size, page_size, _ptr(index), nr_pages, _ptr(pages), n,
                                           _ptr(out), out_stride, _ptr(out_len), _ptr(status), _ptr(workspace),
                                           workspace.numel(), _stream_ptr())
    _check(rc, "csnappy_bc_decompress_pages")
    return out, out_len, status


def bc_decompress_device(d_container, container_length: int | None = None, page_size: int = 4096,
                         out_capacity: int | None = None, *, out=None, result=None, workspace=None):
    """Whole container in device memory -> its pages, page i at out[i * page_size] (the call reads the page count
    back, then enqueues the rest on the current stream).  out_capacity None: out's size, or nr_pages * page_size.
    Returns (out uint8, result int64 [3] = [out_length, rc, failed_page]) CUDA tensors with the values
    bc_decompress_host returns; result[2] is written only when a page fails (default prefilled with -1)."""
    import torch

    n = d_container.numel() if container_length is None else container_length
    dev = d_container.device
    if out_capacity is None:
        if out is not None:
            out_capacity = out.numel()
        else:
            out_capacity = (int.from_bytes(d_container[:4].cpu().numpy().tobytes(), "little") if n >= 4 else 0) * page_size
    if out is None:
        out = torch.empty(max(out_capacity, 1), dtype=torch.uint8, device=dev)
    if result is None:
        result = torch.full((3,), -1, dtype=torch.int64, device=dev)
    words = torch.full((2,), -1, dtype=torch.int32, device=dev)  # status, failed page (u32)
    if workspace is None:
        workspace = _ws(lib().csnappy_bc_decompress_workspace(n, page_size, out_capacity), dev)
    rc = lib().csnappy_bc_decompress(_ptr(d_container), n, page_size, _ptr(out), out_capacity, result.data_ptr(),
                                     words.data_ptr(), words.data_ptr() + 4, _ptr(workspace), workspace.numel(),
                                     _stream_ptr())
    _check(rc, "csnappy_bc_decompress")
    result[1:2].copy_(words[:1])
    failed = words[1:2].to(torch.int64) & 0xFFFFFFFF
    result[2:3].copy_(torch.where(words[1:2] == -1, result[2:3], failed))
    return out, result


def batch_compress(d_in, in_off, in_len, wm: int, *, out_stride: int | None = None):
    """Device-resident batch of csnappy_compress (whole buffers, varint32 header + 32 KiB fragments each).
    d_in: uint8 CUDA tensor; in_off / in_len: HOST sequences (offsets into d_in, lengths).
    Returns (out uint8 [n * out_stride], out_len int32 [n], out_stride)."""
    import torch

    n = len(in_len)
    h_len = np.ascontiguousarray(np.asarray(in_len, dtype=np.uint32))
    h_off = np.ascontiguousarray(np.asarray(in_off, dtype=np.uint64))
    longest = int(h_len.max()) if n else 0
    if out_stride is None:
        out_stride = (5 + longest + longest // 6 + 32 * max(1, -(-longest // FRAGMENT_MAX)) + 15) // 16 * 16
    ws_bytes = lib().csnappy_batch_compress_workspace(h_len.ctypes.data, 0, n)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=d_in.device)
    out = torch.empty(max(n * out_stride, 16), dtype=torch.uint8, device=d_in.device)
    out_len = torch.empty(max(n, 1), dtype=torch.int32, device=d_in.device)
    rc = lib().csnappy_batch_compress(_ptr(d_in), h_off.ctypes.data, 0, h_len.ctypes.data, 0, n, _ptr(out), out_stride,
                                      _ptr(out_len), wm, _ptr(ws), ws_bytes, _stream_ptr())
    _check(rc, "csnappy_batch_compress")
    torch.cuda.current_stream().synchronize()  # the workspace dies with this frame
    return out, out_len, out_stride


def stream_decompress(d_src, src_len: int, out_cap: int, *, out=None, workspace=None, result=None):
    """ONE long raw stream, device resident, through the parallel stream decoder.
    Returns (out uint8 [out_cap], result int32 [2] = [out_len, status]) CUDA tensors (asynchronous)."""
    import torch

    ws_bytes = lib().csnappy_stream_decompress_workspace(src_len, out_cap)
    if workspace is None:
        workspace = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=d_src.device)
    if out is None:
        out = torch.empty(max(out_cap, 16), dtype=torch.uint8, device=d_src.device)
    if result is None:
        result = torch.empty(2, dtype=torch.int32, device=d_src.device)
    rc = lib().csnappy_stream_decompress(_ptr(d_src), src_len, _ptr(out), out_cap, result.data_ptr(),
                                         result.data_ptr() + 4, _ptr(workspace), workspace.numel(), _stream_ptr())
    _check(rc, "csnappy_stream_decompress")
    return out, result


def device_count() -> int:
    return lib().csnappy_b200_device_count()


def set_tuning(key: str, value: int):
    rc = lib().csnappy_b200_set_tuning(key.encode(), value)
    if rc != 0:
        raise ValueError(f"bad tuning {key}={value}")


def kernel_launches() -> int:
    return lib().csnappy_b200_kernel_launches()


def device_ok() -> bool:
    return bool(lib().csnappy_b200_device_ok())


# ----------------------------------------------------------------------------- Snappy framing format
CSNAPPY_E_CHECKSUM = -102
FRAMED_CHUNK = 65536


def framed_max_length(input_length: int) -> int:
    """Exact bound of a framed stream of input_length bytes: 10 + 8 * ceil(n / 65536) + n."""
    return lib().csnappy_framed_max_length(input_length)


def framed_compress(data, wm: int = CSNAPPY_WORKMEM_BYTES_POWER_OF_TWO) -> bytes:
    """Host bytes -> one framed stream (stream identifier, 64 KiB chunks with masked CRC-32C)."""
    n = len(data)
    src = _in_buf(data)
    out = np.empty(framed_max_length(n), dtype=np.uint8)
    olen = C.c_uint64(0)
    rc = lib().csnappy_framed_compress_host(src.ctypes.data, n, out.ctypes.data, out.nbytes, C.byref(olen), wm)
    _check(rc, "csnappy_framed_compress_host")
    return out[: olen.value].tobytes()


def framed_decompress(data, out_capacity: int):
    """Host bytes of a framed stream -> (rc, the valid prefix of the output, failed_offset or None).
    rc: 0, CSNAPPY_E_OUTPUT_INSUF, CSNAPPY_E_DATA_MALFORMED or CSNAPPY_E_CHECKSUM; failed_offset is the header
    position of the failing chunk."""
    src = _in_buf(data)
    out = np.empty(max(out_capacity, 1), dtype=np.uint8)
    olen = C.c_uint64(0)
    bad = C.c_uint64(0)
    rc = lib().csnappy_framed_decompress_host(src.ctypes.data, len(data), out.ctypes.data, out_capacity,
                                              C.byref(olen), C.byref(bad))
    if rc in (CSNAPPY_E_DEVICE, CSNAPPY_E_BAD_ARG):
        _check(rc, "csnappy_framed_decompress_host")
    return rc, out[: olen.value].tobytes(), (bad.value if rc != 0 else None)


def framed_compress_device(d_in, input_length: int | None = None, wm: int = CSNAPPY_WORKMEM_BYTES_POWER_OF_TWO, *,
                           out=None, out_length=None, workspace=None):
    """Device-resident framed compress of a uint8 CUDA tensor, asynchronous on the current stream.
    Returns (out uint8 [framed_max_length(n)], out_length int64 [1]) CUDA tensors."""
    import torch

    n = d_in.numel() if input_length is None else input_length
    cap = framed_max_length(n)
    if out is None:
        out = torch.empty(cap, dtype=torch.uint8, device=d_in.device)
    if out_length is None:
        out_length = torch.empty(1, dtype=torch.int64, device=d_in.device)
    ws_bytes = lib().csnappy_framed_compress_workspace(n)
    if workspace is None:
        workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=d_in.device)
    rc = lib().csnappy_framed_compress(_ptr(d_in), n, _ptr(out), out.numel(), _ptr(out_length), wm, _ptr(workspace),
                                       workspace.numel(), _stream_ptr())
    _check(rc, "csnappy_framed_compress")
    return out, out_length  # the workspace is freed in stream order: the caching allocator reuses it after this work


def framed_decompress_device(d_src, src_length: int | None = None, out_capacity: int = 0, *, out=None, result=None,
                             workspace=None):
    """Device-resident framed decompress, on the current stream (the call waits for the chunk walk, then enqueues
    decoding and verification).  Returns (out uint8 [out_capacity], result int64 [3] = [out_length, rc,
    failed_offset]) CUDA tensors; result[2] is written only when rc != 0."""
    import torch

    n = d_src.numel() if src_length is None else src_length
    if out is None:
        out = torch.empty(max(out_capacity, 1), dtype=torch.uint8, device=d_src.device)
    if result is None:
        result = torch.full((3,), -1, dtype=torch.int64, device=d_src.device)
    ws_bytes = lib().csnappy_framed_decompress_workspace(n)
    if workspace is None:
        workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=d_src.device)
    status = torch.zeros(1, dtype=torch.int32, device=d_src.device)
    rc = lib().csnappy_framed_decompress(_ptr(d_src), n, _ptr(out), out_capacity, result.data_ptr(), status.data_ptr(),
                                         result.data_ptr() + 16, _ptr(workspace), workspace.numel(), _stream_ptr())
    _check(rc, "csnappy_framed_decompress")
    result[1:2].copy_(status)
    return out, result


def framed_crc32c_device(d_in, length: int | None = None, *, crc=None):
    """Masked CRC-32C of each 64 KiB chunk of a uint8 CUDA tensor -> int32 CUDA tensor (as uint32 bits)."""
    import torch

    n = d_in.numel() if length is None else length
    k = -(-n // FRAMED_CHUNK)
    if crc is None:
        crc = torch.empty(max(k, 1), dtype=torch.int32, device=d_in.device)
    rc = lib().csnappy_framed_crc32c(_ptr(d_in), n, _ptr(crc), _stream_ptr())
    _check(rc, "csnappy_framed_crc32c")
    return crc


def _u64(xs) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(xs, dtype=np.uint64).reshape(-1))


def _host_off(a: np.ndarray):
    return a.ctypes.data if a.size else None


def framed_batch_compress_device(d_in, offs, lens, wm: int = CSNAPPY_WORKMEM_BYTES_POWER_OF_TWO, *, out_off=None,
                                 out=None):
    """Many framed streams written in one call: stream i is d_in[offs[i], offs[i] + lens[i]) (HOST sequences).
    Slot i of `out` starts at out_off[i] (None: the running sum of framed_max_length(lens[j]), j < i).
    Returns (out uint8 CUDA tensor, out_off numpy uint64, out_len int64 CUDA tensor), asynchronous on the current
    stream."""
    import torch

    h_off, h_len = _u64(offs), _u64(lens)
    n = len(h_len)
    m = np.array([framed_max_length(int(x)) for x in h_len], dtype=np.uint64)
    h_out = _u64(np.concatenate((np.zeros(1, np.uint64), np.cumsum(m)[:-1]))) if out_off is None else _u64(out_off)
    cap = int((h_out + m).max()) if n else 0
    if out is None:
        out = torch.empty(max(cap, 1), dtype=torch.uint8, device=d_in.device)
    out_len = torch.empty(max(n, 1), dtype=torch.int64, device=d_in.device)
    ws_bytes = lib().csnappy_framed_batch_compress_workspace(_host_off(h_len), n)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=d_in.device)
    rc = lib().csnappy_framed_batch_compress(_ptr(d_in), _host_off(h_off), _host_off(h_len), n, _ptr(out),
                                             None if out_off is None else _host_off(h_out), out.numel(), _ptr(out_len),
                                             wm, _ptr(ws), ws_bytes, _stream_ptr())
    _check(rc, "csnappy_framed_batch_compress")
    return out, h_out, out_len  # the workspace is freed in stream order, as in framed_compress_device


def framed_batch_decompressed_length_device(d_src, offs, lens):
    """Declared decompressed length of every framed stream (the chunk walk, no decoding): returns (length int64,
    status int32) CUDA tensors; status -5 where the walk finds a framing failure (length then counts the chunks before
    it)."""
    import torch

    h_off, h_len = _u64(offs), _u64(lens)
    n = len(h_len)
    length = torch.empty(max(n, 1), dtype=torch.int64, device=d_src.device)
    status = torch.empty(max(n, 1), dtype=torch.int32, device=d_src.device)
    rc = lib().csnappy_framed_batch_decompressed_length(_ptr(d_src), _host_off(h_off), _host_off(h_len), n, _ptr(length),
                                                        _ptr(status), _stream_ptr())
    _check(rc, "csnappy_framed_batch_decompressed_length")
    return length, status


def framed_batch_decompress_device(d_src, offs, lens, caps, *, dst_off=None, dst=None, failed_offset=None):
    """Many framed streams read in one call (the call waits once for the chunk walk of the whole batch).  Output i
    goes to dst[dst_off[i], + caps[i]) (dst_off None: the running sum of caps).  Returns (dst uint8 CUDA tensor,
    dst_off numpy uint64, result int64 CUDA tensor [3, n] = out_len, rc, failed_offset); failed_offset (default
    prefilled with -1) is written only for streams that fail."""
    import torch

    h_off, h_len, h_cap = _u64(offs), _u64(lens), _u64(caps)
    n = len(h_len)
    h_dst = _u64(np.concatenate((np.zeros(1, np.uint64), np.cumsum(h_cap)[:-1]))) if dst_off is None else _u64(dst_off)
    if dst is None:
        dst = torch.empty(max(int((h_dst + h_cap).max()) if n else 0, 1), dtype=torch.uint8, device=d_src.device)
    result = torch.empty((3, max(n, 1)), dtype=torch.int64, device=d_src.device)
    if failed_offset is None:
        result[2].fill_(-1)
    else:
        result[2].copy_(failed_offset)
    status = torch.zeros(max(n, 1), dtype=torch.int32, device=d_src.device)
    ws_bytes = lib().csnappy_framed_batch_decompress_workspace(_host_off(h_len), n)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=d_src.device)
    rc = lib().csnappy_framed_batch_decompress(_ptr(d_src), _host_off(h_off), _host_off(h_len), n, _ptr(dst),
                                               _host_off(h_dst), _host_off(h_cap), result[0].data_ptr(), _ptr(status),
                                               result[2].data_ptr(), _ptr(ws), ws_bytes, _stream_ptr())
    _check(rc, "csnappy_framed_batch_decompress")
    result[1].copy_(status)
    return dst, h_dst, result


def _stage(bufs):
    """Byte strings -> (one uint8 CUDA tensor, offsets, lengths)."""
    import torch

    lens = [len(b) for b in bufs]
    offs = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.uint64) if bufs else np.zeros(0, np.uint64)
    host = np.frombuffer(b"".join(bytes(b) for b in bufs) or b"\0", dtype=np.uint8)
    return torch.from_numpy(host.copy()).cuda(), offs, lens


def framed_batch_compress(bufs, wm: int = CSNAPPY_WORKMEM_BYTES_POWER_OF_TWO) -> list[bytes]:
    """A list of byte strings -> their framed streams, written in one device call."""
    import torch

    if not bufs:
        return []
    d, offs, lens = _stage(bufs)
    out, out_off, out_len = framed_batch_compress_device(d, offs, lens, wm)
    torch.cuda.current_stream().synchronize()
    raw, ol = out.cpu().numpy(), out_len.cpu().tolist()
    return [raw[int(o):int(o) + n].tobytes() for o, n in zip(out_off, ol)]


def framed_batch_decompress(bufs, caps=None):
    """A list of framed streams -> [(rc, valid prefix, failed_offset or None)], read in one device call.  caps=None:
    each stream's capacity is its declared length (framed_batch_decompressed_length_device)."""
    import torch

    if not bufs:
        return []
    d, offs, lens = _stage(bufs)
    if caps is None:
        length, _ = framed_batch_decompressed_length_device(d, offs, lens)
        caps = length[: len(bufs)].cpu().tolist()
    dst, dst_off, res = framed_batch_decompress_device(d, offs, lens, caps)
    torch.cuda.current_stream().synchronize()
    raw, r = dst.cpu().numpy(), res.cpu().tolist()
    return [(int(r[1][i]), raw[int(dst_off[i]):int(dst_off[i]) + r[0][i]].tobytes(), r[2][i] if r[1][i] else None)
            for i in range(len(bufs))]
