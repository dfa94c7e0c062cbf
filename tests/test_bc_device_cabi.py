"""The device-buffer page container calls at the C-ABI boundary without a GPU: the workspace arithmetic, refused
arguments coming before any device work, and the calls failing loudly (CSNAPPY_E_DEVICE) rather than falling back when
no device is present."""
import ctypes as C

import pytest

NONE = 2**64 - 1
E_DEVICE, E_BAD_ARG = -100, -101


@pytest.fixture(scope="module")
def lib():
    from csnappy_b200 import build

    build.build()
    from csnappy_b200._lib import lib as load

    return load()


def slot(page):
    return (32 + page + page // 6 + 15) // 16 * 16


def test_compress_workspace(lib):
    for page in (1, 13, 4095, 4096, 32768):
        prev = 0
        for n in sorted({0, 1, page - 1, page, page + 1, 1000 * page + 3, 2**20 * page}):
            ws = lib.csnappy_bc_compress_workspace(n, page)
            nr = -(-n // page)
            assert ws >= nr * slot(page) + 16 * nr and ws > 0, (page, n)
            assert ws >= prev, (page, n)
            prev = ws
        assert lib.csnappy_bc_compress_workspace((2**32 - 1) * page, page) < NONE
        assert lib.csnappy_bc_compress_workspace((2**32 - 1) * page + 1, page) == NONE
    assert lib.csnappy_bc_compress_workspace(100, 0) == NONE
    assert lib.csnappy_bc_compress_workspace(100, 32769) == NONE


def test_page_read_workspace(lib):
    prev = 0
    for n in (0, 1, 2, 1000, 100_000, 2**32 - 1):
        ws = lib.csnappy_bc_decompress_pages_workspace(n)
        assert ws >= 16 * n and ws >= prev
        prev = ws


def test_whole_read_workspace(lib):
    for page in (1, 1000, 4096, 32768):
        prev = 0
        for length in (0, 3, 4, 8, 4 + 4 * 1000, 10**9, 2**40):
            ws = lib.csnappy_bc_decompress_workspace(length, page, 2**50)
            pages = max(length - 4, 0) // 4 if length >= 4 else 0
            assert ws >= 20 * min(pages, 2**32 - 1) and ws >= prev, (page, length)
            prev = ws
        # bounded by the output's pages too
        assert lib.csnappy_bc_decompress_workspace(2**40, page, 10 * page) == lib.csnappy_bc_decompress_workspace(
            4 + 40, page, 2**50)
        assert lib.csnappy_bc_decompress_workspace(2**50, page, 2**62) < NONE
    assert lib.csnappy_bc_decompress_workspace(1000, 0, 1000) == NONE
    assert lib.csnappy_bc_decompress_workspace(1000, 32769, 1000) == NONE


def test_refused_arguments_and_no_fallback(lib):
    import torch

    buf = C.create_string_buffer(1 << 20)
    p = C.addressof(buf)
    ws = 1 << 19
    nr = C.c_uint32(0)
    cap = lib.csnappy_bc_max_container_length(1000, 100)
    # writer: wm, page size, capacity, workspace, null buffers
    assert lib.csnappy_bc_compress(p, 1000, 100, p, cap, p, 8, p, ws, None) == E_BAD_ARG
    assert lib.csnappy_bc_compress(p, 1000, 0, p, cap, p, 13, p, ws, None) == E_BAD_ARG
    assert lib.csnappy_bc_compress(p, 1000, 32769, p, cap, p, 13, p, ws, None) == E_BAD_ARG
    assert lib.csnappy_bc_compress(p, 1000, 100, p, cap - 1, p, 13, p, ws, None) == E_BAD_ARG
    need = lib.csnappy_bc_compress_workspace(1000, 100)
    assert lib.csnappy_bc_compress(p, 1000, 100, p, cap, p, 13, p, need - 1, None) == E_BAD_ARG
    assert lib.csnappy_bc_compress(None, 1000, 100, p, cap, p, 13, p, ws, None) == E_BAD_ARG
    assert lib.csnappy_bc_compress(p, 2**32 * 100, 100, p, 2**60, p, 13, p, ws, None) == E_BAD_ARG
    # index: page size, short header, index without storage
    assert lib.csnappy_bc_index(p, 100, 0, p, 10, C.byref(nr), None) == E_BAD_ARG
    assert lib.csnappy_bc_index(p, 3, 100, p, 10, C.byref(nr), None) == E_BAD_ARG
    assert lib.csnappy_bc_index(p, 100, 100, None, 10, C.byref(nr), None) == E_BAD_ARG
    assert lib.csnappy_bc_index(p, 100, 100, p, 10, None, None) == E_BAD_ARG
    # page reads: stride, container shorter than the index of nr_pages, workspace, null buffers; 0 requests: nothing
    wsp = lib.csnappy_bc_decompress_pages_workspace(10)
    assert lib.csnappy_bc_decompress_pages(p, 4000, 100, p, 10, p, 10, p, 99, p, p, p, wsp, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress_pages(p, 43, 100, p, 10, p, 10, p, 100, p, p, p, wsp, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress_pages(p, 4000, 100, p, 10, p, 10, p, 100, p, p, p, wsp - 1, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress_pages(p, 4000, 100, p, 10, None, 10, p, 100, p, p, p, wsp, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress_pages(p, 4000, 100, p, 10, p, 0, p, 100, p, p, p, 0, None) == 0
    # whole container: page size, short header, workspace, null buffers
    wsd = lib.csnappy_bc_decompress_workspace(4000, 100, 100000)
    assert lib.csnappy_bc_decompress(p, 4000, 0, p, 100000, p, p, p, p, ws, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress(p, 3, 100, p, 100000, p, p, p, p, ws, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress(p, 4000, 100, p, 100000, p, p, p, p, wsd - 1, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress(p, 4000, 100, None, 100000, p, p, p, p, wsd, None) == E_BAD_ARG
    assert lib.csnappy_bc_decompress(p, 4000, 100, p, 100000, None, p, p, p, wsd, None) == E_BAD_ARG
    if torch.cuda.is_available():
        return  # the no-device behaviour cannot be observed
    # accepted arguments without a device: CSNAPPY_E_DEVICE, no fallback
    assert lib.csnappy_bc_compress(p, 1000, 100, p, cap, p, 13, p, ws, None) == E_DEVICE
    assert b"csnappy_b200" in lib.csnappy_b200_last_error()
    assert lib.csnappy_bc_index(p, 4000, 100, p, 10, C.byref(nr), None) == E_DEVICE
    assert lib.csnappy_bc_decompress_pages(p, 4000, 100, p, 10, p, 10, p, 100, p, p, p, wsp, None) == E_DEVICE
    assert lib.csnappy_bc_decompress(p, 4000, 100, p, 100000, p, p, p, p, wsd, None) == E_DEVICE
