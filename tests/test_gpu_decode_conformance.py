"""Every GPU decode path against streams whose result is known by construction (tests/streams.py).

The other GPU decode tests feed csnappy's own compressor output and corruptions of it, which use a narrow part
of the format.  Here the batched decoder (staged, input through L1, global and lane-per-block paths, every
lane group), the drop-in calls and the parallel single-stream decoder decode every tag form: copy-4 tags,
copies of 1-3 bytes, offsets at every class and output phase, literals with 1-4 length bytes, the zero-length
literal, headers across the stream decoder's 4 KiB input chunks, inputs longer than max_compressed_length(cap),
and invalid streams with their first failing tag.  Status, length and bytes must equal the construction, and
nothing at or past a block's capacity may change (every output slot is pre-filled with a pattern, and a 256-byte
guard band follows it).  test_stream_conformance.py checks the same streams against the CPU oracle port.
"""
import hashlib
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import streams as S  # noqa: E402

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAT = 0xA5
GUARD = 256
BIN_EDGES = (640, 4736, 34048, 1 << 20)  # blocks are grouped by capacity, so that the output slots stay small


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.fixture(scope="module")
def bins():
    cases = S.copy_matrix(201) + S.large_copy_matrix(202) + S.boundary_streams(203) + S.invalid_cases(204) + \
        S.overlong_streams(205)
    cases += [S.Case(S.random_stream(k, 4096), name="random 4 KiB") for k in range(40)]
    cases += [S.Case(S.random_stream(100 + k, 32768), name="random 32 KiB") for k in range(8)]
    out = []
    lo = 0
    for hi in BIN_EDGES:
        b = [c for c in cases if lo <= c.cap < hi]
        assert b
        out.append(b)
        lo = hi
    assert sum(map(len, out)) == len(cases)
    return out


def _sha(b):
    return hashlib.sha256(b).hexdigest()


def _expected(cases, caps, stride):
    """(expected slots, mask of the bytes that must match, status, out_len) for `cases` decoded into `caps`."""
    B = len(cases)
    exp = np.full((B, stride), PAT, dtype=np.uint8)
    mask = np.zeros((B, stride), dtype=bool)
    st = np.zeros(B, dtype=np.int32)
    ol = np.zeros(B, dtype=np.int64)
    for i, c in enumerate(cases):
        rc, _, out = c.expect(caps[i])
        st[i] = rc
        if rc == 0:
            ol[i] = len(out)
            exp[i, : len(out)] = np.frombuffer(out, dtype=np.uint8)
            mask[i, : len(out)] = True
        mask[i, caps[i]:] = True  # nothing at or past the capacity changes
    return exp, mask, st, ol


def _inputs(cases, layout, prefix=None):
    datas = [prefix(c) if prefix else c.data for c in cases]
    lens = torch.tensor([len(d) for d in datas], dtype=torch.int32).cuda()
    if layout == "stride":
        in_stride = (max(len(d) for d in datas) + 16 + 15) // 16 * 16
        host = np.zeros((len(datas), in_stride), dtype=np.uint8)
        for i, d in enumerate(datas):
            host[i, : len(d)] = np.frombuffer(d, dtype=np.uint8)
        return torch.from_numpy(host.reshape(-1)).cuda(), lens, dict(in_stride=in_stride)
    # back to back from an odd address: every block at its own alignment
    offs = np.zeros(len(datas), dtype=np.int64)
    pos = 1
    for i, d in enumerate(datas):
        offs[i] = pos
        pos += len(d)
    host = np.zeros(pos + 64, dtype=np.uint8)
    for i, d in enumerate(datas):
        host[offs[i]: offs[i] + len(d)] = np.frombuffer(d, dtype=np.uint8)
    return torch.from_numpy(host).cuda(), lens, dict(in_off=torch.from_numpy(offs).cuda())


def _decode_and_check(cs, cases, caps, layout, uniform):
    B = len(cases)
    stride = (max(caps) + GUARD + 15) // 16 * 16
    d_in, d_len, kw = _inputs(cases, layout)
    out = torch.full((B * stride + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    if uniform:
        assert len(set(caps)) == 1
        kw["out_caps"] = None
    else:
        kw["out_caps"] = torch.tensor(caps, dtype=torch.int32).cuda()
    _, out_len, status = cs.batch_decompress(d_in, d_len, B, caps[0], out=out, out_stride=stride, **kw)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert (o[B * stride:] == PAT).all(), "wrote past the last slot"
    got = o[: B * stride].reshape(B, stride)
    exp, mask, st, ol = _expected(cases, caps, stride)
    got_st, got_ol = status.cpu().numpy()[:B], out_len.cpu().numpy()[:B].astype(np.int64)
    wrong = np.nonzero(got_st != st)[0]
    assert not len(wrong), [(cases[i].name, int(got_st[i]), int(st[i])) for i in wrong[:8]]
    ok = st == 0
    wrong = np.nonzero(ok & (got_ol != ol))[0]
    assert not len(wrong), [(cases[i].name, int(got_ol[i]), int(ol[i])) for i in wrong[:8]]
    wrong = np.nonzero(((got != exp) & mask).any(axis=1))[0]
    assert not len(wrong), [(cases[i].name, caps[i], int(st[i]),
                             int(np.nonzero((got[i] != exp[i]) & mask[i])[0][0])) for i in wrong[:8]]


# (decompress_lanes, decompress_stage_input, decompress_lane_warps): staged, input through L1, global, lane decoder
CONFIGS = [(g, stage, 0) for g in (8, 16, 32) for stage in (1, 2, 3)] + [(32, 4, 0), (32, 4, 1)]


@pytest.mark.parametrize("uniform", [False, True], ids=["per_block_caps", "uniform_cap"])
@pytest.mark.parametrize("layout", ["stride", "packed"])
@pytest.mark.parametrize("lanes,stage,warps", CONFIGS)
def test_batch_decompress_conformance(cs, bins, lanes, stage, warps, layout, uniform):
    cs.set_tuning("decompress_lanes", lanes)
    cs.set_tuning("decompress_stage_input", stage)
    cs.set_tuning("decompress_lane_warps", warps)
    try:
        for cases in bins:
            caps = [max(c.cap for c in cases)] * len(cases) if uniform else [c.cap for c in cases]
            _decode_and_check(cs, cases, caps, layout, uniform)
    finally:
        cs.set_tuning("decompress_lanes", 0)
        cs.set_tuning("decompress_stage_input", 0)
        cs.set_tuning("decompress_lane_warps", 0)


@pytest.mark.parametrize("stage", [1, 3, 4])
def test_batch_decompress_with_header_conformance(cs, bins, stage):
    """BATCH_WITH_HEADER: the varint32 length becomes the capacity; a length above the caller's is -2, a bad
    header -1.  Nothing past the caller's capacity changes."""
    rng = np.random.default_rng(stage)
    cases = [c for b in bins[:2] for c in b if c.end is None and c.s.produced <= 4096][::5]
    pick = rng.random(len(cases))
    # caller capacity: the stated length, more, or one byte less (-2)
    caps = [c.s.produced + (0 if p < 0.5 else (64 if p < 0.8 else -1)) for c, p in zip(cases, pick)]
    caps = [max(x, 0) for x in caps]
    cs.set_tuning("decompress_stage_input", stage)
    try:
        B = len(cases)
        stride = (max(caps) + GUARD + 15) // 16 * 16
        d_in, d_len, kw = _inputs(cases, "packed", lambda c: c.s.with_header())
        out = torch.full((B * stride + GUARD,), PAT, dtype=torch.uint8, device="cuda")
        _, out_len, status = cs.batch_decompress(d_in, d_len, B, 0, out=out, out_stride=stride,
                                                 out_caps=torch.tensor(caps, dtype=torch.int32).cuda(),
                                                 flags=cs.api.BATCH_WITH_HEADER, **kw)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("decompress_stage_input", 0)
    o = out.cpu().numpy()
    assert (o[B * stride:] == PAT).all()
    st, ol = status.cpu().numpy(), out_len.cpu().numpy()
    n_insuf = 0
    for i, c in enumerate(cases):
        slot = o[i * stride:(i + 1) * stride]
        assert (slot[caps[i]:] == PAT).all(), (c.name, "wrote at or past cap")
        if c.s.produced > caps[i]:
            assert st[i] == cs.CSNAPPY_E_OUTPUT_INSUF, c.name
            n_insuf += 1
            continue
        rc, _, exp = c.s.expect(c.s.produced)
        assert st[i] == rc, (c.name, int(st[i]), rc)
        if rc == 0:
            assert ol[i] == len(exp) and slot[: ol[i]].tobytes() == exp, c.name
    assert n_insuf > 10


def test_batch_decompress_bad_headers(cs):
    hdrs = [b"", b"\xff\xff\xff\xff\xff\x00", b"\x80", b"\x85\x80"]
    B = len(hdrs)
    host = np.zeros((B, 16), dtype=np.uint8)
    for i, h in enumerate(hdrs):
        host[i, : len(h)] = np.frombuffer(h, dtype=np.uint8)
    lens = torch.tensor([len(h) for h in hdrs], dtype=torch.int32).cuda()
    _, _, status = cs.batch_decompress(torch.from_numpy(host.reshape(-1)).cuda(), lens, B, 64, in_stride=16,
                                       flags=cs.api.BATCH_WITH_HEADER)
    torch.cuda.synchronize()
    assert status.cpu().numpy()[:B].tolist() == [cs.CSNAPPY_E_HEADER_BAD] * B


def test_dropin_decompress_conformance(cs, bins):
    """csnappy_decompress_noheader / csnappy_decompress (streams up to 64 KiB: one block through the batched decoder)."""
    rng = np.random.default_rng(5)
    cases = [c for b in bins for c in b if len(c.data) <= 65536 and c.cap <= 65536]
    idx = rng.choice(len(cases), 500, replace=False)
    sample = [cases[i] for i in idx] + [c for c in cases if "header cut" in c.name or "2^31" in c.name][:150]
    for c in sample:
        rc, _, exp = c.expect()
        got_rc, got = cs.csnappy_decompress_noheader(c.data, c.cap)
        assert got_rc == rc, (c.name, got_rc, rc)
        if rc == 0:
            assert got == exp, c.name
    for c in sample[:150]:
        if c.end is not None:
            continue
        n = c.s.produced
        rc, _, exp = c.s.expect(n)
        got_rc, got = cs.csnappy_decompress(c.s.with_header(), c.cap)
        if n > c.cap:
            assert got_rc == cs.CSNAPPY_E_OUTPUT_INSUF, c.name
        else:
            assert got_rc == rc, c.name
            if rc == 0:
                assert got[:n] == exp, c.name


@pytest.fixture(scope="module")
def long_cases():
    """Multi-MiB streams: valid, one byte short of space, cut off, with a bad offset near the end; expected digests."""
    cases = []
    for seed, n in ((11, 3 << 20), (12, 16 << 20)):
        s = S.long_stream(seed, n)
        cases += [S.Case(s, name=f"long {n}"), S.Case(s, cap=s.produced - 1, name=f"long {n}, cap - 1"),
                  S.Case(s, end=len(s.buf) - 3, name=f"long {n}, cut")]
    s = S.long_stream(13, 2 << 20)
    s.copy(s.produced + 1, 9, 4).lit(b"tail")
    cases.append(S.Case(s, name="long, bad offset at the end"))
    s = S.random_stream(14, 1 << 20)
    cases.append(S.Case(s, name="random 1 MiB"))
    exp = []
    for c in cases:
        rc, _, out = c.expect()
        exp.append((rc, _sha(out) if rc == 0 else None, len(out) if rc == 0 else 0))
    return cases, exp


@pytest.mark.parametrize("stream_min", [0, -1], ids=["parallel", "serial"])
def test_dropin_long_streams(cs, long_cases, stream_min):
    cases, exp = long_cases
    cs.set_tuning("stream_decode_min", stream_min)
    try:
        for c, (rc, digest, _) in zip(cases, exp):
            got_rc, got = cs.csnappy_decompress_noheader(c.data, c.cap)
            assert got_rc == rc, (c.name, got_rc, rc)
            if rc == 0:
                assert _sha(got) == digest, c.name
    finally:
        cs.set_tuning("stream_decode_min", 0)


def _stream_decompress(cs, data: bytes, cap: int):
    d_src = torch.zeros(max(len(data), 1) + 64, dtype=torch.uint8, device="cuda")
    if data:
        d_src[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    out = torch.full((cap + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    _, result = cs.api.stream_decompress(d_src, len(data), cap, out=out)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert (o[cap:] == PAT).all(), "wrote at or past cap"
    out_len, status = result.cpu().numpy().tolist()
    return status, out_len, o


def test_stream_decompress_device_entry(cs, long_cases):
    """csnappy_stream_decompress: the empty stream (the serial fallback), input lengths around one 4 KiB chunk,
    and the multi-MiB streams."""
    status, out_len, _ = _stream_decompress(cs, b"", 100)
    assert (status, out_len) == (0, 0)
    cases = []
    for n in (2, 100, 4095, 4096, 4097, 8192, 8193):
        s = S.stream_of_input_len(300 + n, n)
        assert len(s.buf) == n
        cases += [S.Case(s, name=f"{n} input bytes"), S.Case(s, cap=s.produced - 1, name=f"{n} input bytes, cap - 1"),
                  S.Case(s, end=n - 1, name=f"{n} input bytes, cut")]
    for c in cases:
        rc, _, exp = c.expect()
        status, out_len, o = _stream_decompress(cs, c.data, c.cap)
        assert status == rc, (c.name, status, rc)
        if rc == 0:
            assert out_len == len(exp) and o[:out_len].tobytes() == exp, c.name
    for c, (rc, digest, n) in zip(*long_cases):
        status, out_len, o = _stream_decompress(cs, c.data, c.cap)
        assert status == rc, (c.name, status, rc)
        if rc == 0:
            assert out_len == n and _sha(o[:n].tobytes()) == digest, c.name
