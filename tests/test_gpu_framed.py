"""The framing format on the device against the restatement (tests/framed.py): writer bytes at every wm, the reader's
(rc, out_length, failed_offset) and prefix on every hostile stream, guard bands, the device and host calls, refused
arguments, the CRC kernel at every length and alignment, and a round trip of more than 1 GiB."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

import framed as F
import oracle
import streams

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from csnappy_b200 import api  # noqa: E402
from csnappy_b200._lib import lib  # noqa: E402

GUARD = 4096


@pytest.fixture(scope="module")
def hostile():
    return F.hostile_streams(11, 16, stream_cases=streams.boundary_streams(7)[::3] + streams.copy_matrix(7, phases=(0,))[::60])


def _host_decompress(src: bytes, cap: int, offset: int = 0, pinned: bool = False):
    """The host call with the output at `offset` in a buffer with a guard band behind out_capacity."""
    n = offset + cap + GUARD
    if pinned:
        t = torch.full((n,), 0xA5, dtype=torch.uint8).pin_memory()
        buf, ptr = t, t.data_ptr()
        s = torch.empty(len(src) + 16, dtype=torch.uint8).pin_memory()
        s[3:3 + len(src)] = torch.frombuffer(bytearray(src), dtype=torch.uint8) if src else s[3:3]
        sptr = s.data_ptr() + 3
    else:
        buf = np.full(n, 0xA5, dtype=np.uint8)
        ptr = buf.ctypes.data
        sarr = np.frombuffer(b"\0\0\0" + bytes(src) + b"\0", dtype=np.uint8).copy()
        sptr = sarr.ctypes.data + 3
    olen, bad = C.c_uint64(0), C.c_uint64(0xDEAD)
    rc = lib().csnappy_framed_decompress_host(sptr, len(src), ptr + offset, cap, C.byref(olen), C.byref(bad))
    raw = bytes(buf.numpy()) if pinned else buf.tobytes()
    assert raw[offset + cap:] == b"\xa5" * GUARD, "bytes behind out_capacity were written"
    assert raw[:offset] == b"\xa5" * offset
    return rc, olen.value, (bad.value if rc else None), raw[offset:offset + olen.value]


def _check_read(got, exp: F.ReadResult, what):
    rc, olen, bad, data = got
    assert (rc, olen, bad) == exp.key(), what
    assert data == exp.data, what


# ---------------------------------------------------------------------------------------------------- writer
FUZZ = [(F.mixed_bytes(s, n, scale=sc)) for s, n, sc in ((1, 200000, 5000), (2, 300001, 70000), (3, 65536 * 3, 300))]


@pytest.mark.parametrize("wm", range(9, 17))
def test_compress_matches_restatement(wm):
    port = oracle.port()
    inputs = list(FUZZ) + [F.mixed_bytes(n + 1, n, scale=9000) for n in F.LENGTHS if n < 2**20 or wm in (9, 16)]
    for data in inputs:
        assert api.framed_compress(data, wm) == F.write_framed(data, wm, port), (len(data), wm)


@pytest.mark.parametrize("n", [F.CHUNK, 4096])
def test_compress_type_rule_edge(n):
    port = oracle.port()
    for d in (-1, 0, 1):
        c = F.edge_chunk(n, 16, d, port=port)
        pre = F.mixed_bytes(9, F.CHUNK if n < F.CHUNK else 0)  # the 4096-byte edge chunk as the short last chunk
        data = pre + c
        assert api.framed_compress(data, 16) == F.write_framed(data, 16, port), d


def test_compress_device_guard_and_alignment():
    for off in (0, 1, 3, 7):
        data = F.mixed_bytes(off, 150000 + off, scale=3000)
        d = torch.empty(len(data) + 8, dtype=torch.uint8, device="cuda")
        d[off:off + len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        cap = F.max_length(len(data))
        out = torch.full((cap + 1 + GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        o, olen = api.framed_compress_device(d[off:], len(data), 14, out=out[1:])
        torch.cuda.synchronize()
        raw = bytes(out.cpu().numpy())
        exp = F.write_framed(data, 14)
        assert int(olen.item()) == len(exp)
        assert raw[1:1 + len(exp)] == exp
        assert raw[0] == 0xA5 and raw[1 + cap:] == b"\xa5" * GUARD


# ---------------------------------------------------------------------------------------------------- reader
def test_reader_on_hostile_streams_host(hostile):
    for i, h in enumerate(hostile):
        exp = F.read_framed(h.stream, h.cap)
        _check_read(_host_decompress(h.stream, h.cap, offset=i % 5), exp, h.cls)


def test_reader_on_hostile_streams_device(hostile):
    for h in hostile[::3]:
        exp = F.read_framed(h.stream, h.cap)
        src = torch.frombuffer(bytearray(h.stream + b"\0"), dtype=torch.uint8).cuda()
        out = torch.full((h.cap + 3 + GUARD,), 0xA5, dtype=torch.uint8, device="cuda")
        o, res = api.framed_decompress_device(src, len(h.stream), h.cap, out=out[3:])
        torch.cuda.synchronize()
        r = res.cpu().tolist()
        assert (int(r[1]), r[0], r[2] if r[1] else None) == exp.key(), h.cls
        raw = bytes(out.cpu().numpy())
        assert raw[3:3 + exp.out_length] == exp.data, h.cls
        assert raw[:3] == b"\xa5" * 3 and raw[3 + h.cap:] == b"\xa5" * GUARD, h.cls


@pytest.mark.parametrize("stage", [1, 2, 3, 4])
def test_reader_every_decoder_path(hostile, stage):
    """out_off through every routing of the batched decoder (staged, output-staged, global, lane-per-block asked)."""
    pick = [h for h in hostile if h.cls in ("foreign_chunking", "valid", "two_failures_decode_crc")]
    pick += [h for h in hostile if h.cls == "tag_forms"][::8]
    api.set_tuning("decompress_stage_input", stage)
    try:
        for h in pick:
            _check_read(_host_decompress(h.stream, h.cap, offset=1), F.read_framed(h.stream, h.cap), h.cls)
    finally:
        api.set_tuning("decompress_stage_input", 0)


def test_truncation_at_every_byte_of_a_small_stream():
    data = F.mixed_bytes(5, 1500, scale=100)
    s = F.write_framed(data, 16)
    for end in range(len(s) + 1):
        _check_read(_host_decompress(s[:end], len(data)), F.read_framed(s[:end], len(data)), end)


@pytest.mark.parametrize("pinned", [False, True])
def test_host_round_trip_pinned_and_pageable(pinned):
    for n in F.LENGTHS:
        data = F.mixed_bytes(n, n, scale=40000)
        s = api.framed_compress(data, 16)
        for off in (0, 1, 5):
            rc, olen, bad, out = _host_decompress(s, n + off, offset=off, pinned=pinned)
            assert (rc, olen, bad, out) == (0, n, None, data)


def test_refused_arguments():
    L = lib()
    buf = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    p, ws = buf.data_ptr(), buf.data_ptr() + (1 << 19)
    s = torch.cuda.current_stream().cuda_stream
    wsc = L.csnappy_framed_compress_workspace(1000)
    cap = L.csnappy_framed_max_length(1000)
    assert cap == 1018
    ok = L.csnappy_framed_compress(p, 1000, p + 4096, cap, p + 8192, 16, ws, wsc, s)
    assert ok == 0
    for args in ((p, 1000, p + 4096, cap, p + 8192, 8, ws, wsc, s),
                 (p, 1000, p + 4096, cap, p + 8192, 17, ws, wsc, s),
                 (p, 1000, p + 4096, cap - 1, p + 8192, 16, ws, wsc, s),
                 (p, 1000, p + 4096, cap, p + 8192, 16, ws, wsc - 1, s),
                 (None, 1000, p + 4096, cap, p + 8192, 16, ws, wsc, s),
                 (p, 1000, None, cap, p + 8192, 16, ws, wsc, s),
                 (p, 1000, p + 4096, cap, None, 16, ws, wsc, s),
                 (p, 1000, p + 4096, cap, p + 8192, 16, None, wsc, s)):
        assert L.csnappy_framed_compress(*args) == api.CSNAPPY_E_BAD_ARG, args
    wsd = L.csnappy_framed_decompress_workspace(1000)
    for args in ((p, 1000, p + 4096, 10, p + 8192, p + 8200, p + 8208, ws, wsd - 1, s),
                 (None, 1000, p + 4096, 10, p + 8192, p + 8200, p + 8208, ws, wsd, s),
                 (p, 1000, None, 10, p + 8192, p + 8200, p + 8208, ws, wsd, s),
                 (p, 1000, p + 4096, 10, None, p + 8200, p + 8208, ws, wsd, s),
                 (p, 1000, p + 4096, 10, p + 8192, None, p + 8208, ws, wsd, s)):
        assert L.csnappy_framed_decompress(*args) == api.CSNAPPY_E_BAD_ARG, args
    h = np.zeros(4096, dtype=np.uint8)
    n = C.c_uint64(0)
    assert L.csnappy_framed_compress_host(h.ctypes.data, 100, h.ctypes.data, 117, C.byref(n), 16) == api.CSNAPPY_E_BAD_ARG
    assert L.csnappy_framed_compress_host(h.ctypes.data, 100, h.ctypes.data, 118, C.byref(n), 9) == 0
    assert L.csnappy_framed_compress_host(h.ctypes.data, 100, h.ctypes.data, 118, C.byref(n), 8) == api.CSNAPPY_E_BAD_ARG
    assert L.csnappy_framed_compress_host(None, 100, h.ctypes.data, 118, C.byref(n), 16) == api.CSNAPPY_E_BAD_ARG
    assert L.csnappy_framed_decompress_host(None, 100, h.ctypes.data, 10, C.byref(n), None) == api.CSNAPPY_E_BAD_ARG
    assert L.csnappy_framed_decompress_host(h.ctypes.data, 100, None, 10, C.byref(n), None) == api.CSNAPPY_E_BAD_ARG
    assert L.csnappy_framed_decompress_host(h.ctypes.data, 100, h.ctypes.data, 10, None, None) == api.CSNAPPY_E_BAD_ARG
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- CRC kernel
def test_crc_kernel_every_length_and_alignment():
    rng = np.random.default_rng(17)
    src = rng.integers(0, 256, F.CHUNK + 64, dtype=np.uint8)
    d = torch.from_numpy(src).cuda()
    lengths = list(range(0, 1025)) + [int(x) for x in rng.integers(1025, F.CHUNK + 1, 60)] + [F.CHUNK]
    out = torch.zeros(len(lengths) * 16, dtype=torch.int32, device="cuda")
    bufs = []
    for i, n in enumerate(lengths):
        for a in range(16):
            api.framed_crc32c_device(d[a:], n, crc=out[i * 16 + a:])
            bufs.append(src[a:a + n].tobytes())
    got = (out.cpu().numpy().view(np.uint32)).tolist()
    exp = [F.mask(c) if b else 0 for c, b in zip(F.crc32c_many(bufs), bufs)]  # an empty buffer has no chunk: no write
    bad = [(lengths[k // 16], k % 16) for k in range(len(bufs)) if got[k] != exp[k]]
    assert not bad, bad[:10]


def test_crc_kernel_many_chunks():
    data = F.mixed_bytes(8, 5 * F.CHUNK + 1234)
    crc = api.framed_crc32c_device(torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda())
    chunks = [data[i:i + F.CHUNK] for i in range(0, len(data), F.CHUNK)]
    assert crc.cpu().numpy().view(np.uint32).tolist() == [F.mask(c) for c in F.crc32c_many(chunks)]


# ---------------------------------------------------------------------------------------------------- large
def test_round_trip_above_1_gib():
    n = (1 << 30) + 12345
    g = torch.Generator(device="cuda").manual_seed(3)
    d = torch.randint(97, 101, (n,), dtype=torch.uint8, device="cuda", generator=g)
    d[: n // 3] = torch.randint(0, 256, (n // 3,), dtype=torch.uint8, device="cuda", generator=g)
    s, slen = api.framed_compress_device(d, n, 16)
    slen = int(slen.item())
    out, res = api.framed_decompress_device(s, slen, n)
    torch.cuda.synchronize()
    assert res[:2].cpu().tolist() == [n, 0]
    assert torch.equal(out[:n], d)
    # one flipped bit deep inside fails that chunk with the checksum and keeps every chunk before it
    k = 3000
    hdr = 10 + 0  # find chunk k's position on the host from the headers
    sh = s[:slen].cpu().numpy()
    pos = hdr
    for _ in range(k):
        pos += 4 + int(sh[pos + 1]) + (int(sh[pos + 2]) << 8) + (int(sh[pos + 3]) << 16)
    assert sh[pos] == 1  # random chunks are stored
    s[pos + 100] ^= 1
    out, res = api.framed_decompress_device(s, slen, n)
    torch.cuda.synchronize()
    assert res.cpu().tolist() == [k * F.CHUNK, api.CSNAPPY_E_CHECKSUM, pos]
