"""The parallel single-stream decoder (stream_kernel.cu, csnappy_stream_decompress) against streams whose result is
known by construction, at every input-chunk phase that matters, and every decoder at capacities of 2 GiB and above.

The stream decoder ranks tag lists inside 4096-byte input chunks, hops from chunk to chunk with one thread, and
reports the failing tag with the smallest input position.  Here it decodes (tests/stream_chunks.py):

  * the whole invalid corpus of tests/streams.py with a chunk boundary before each byte of the failing tag's header;
  * the boundary, large-copy and overlong streams with a boundary before, inside the header of and inside the
    payload of their last tag, and every 8th copy-matrix stream at two phases;
  * streams built on the chunk grid: literals over whole chunks, a chunk entered at its last byte, a chunk of 2048
    copy-1 tags failing at chosen tag indices, failures in two chunks, inputs of one byte around whole chunks.

A shifted case decodes to the unshifted case's result (test_stream_chunks.py pins that on the CPU).  Each call gets
its own output slot, pre-filled with a pattern and followed by a 256-byte guard band: status, length and bytes must
equal the construction, and nothing at or past the capacity may change.

Capacities of 2^31 and above: a literal whose length is 2^31 or more passes the reference's signed payload test, so
with room for its length the result is -5, not -3.  Every decoder is checked there, and the stream decoder writes a
2^31 + 2^20 byte output whose copy-4 offsets exceed 2^31.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import stream_chunks as C  # noqa: E402
import streams as S  # noqa: E402

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAT = 0xA5
GUARD = 256
BIG = (1 << 31) + (1 << 20)


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.fixture(scope="module")
def plan():
    return C.shift_plan()


def _to_device(data: bytes):
    t = torch.empty(len(data) + 64, dtype=torch.uint8)
    t[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8)
    t[len(data):] = 0
    return t.cuda()


def _stream_calls(cs, calls):
    """calls: (name, input bytes, cap, expected (rc, _, out)).  Every call is enqueued on the current stream with one
    shared workspace (the calls are ordered on that stream), the stream is synchronised once, then every status,
    length, output and guard band is checked."""
    n = len(calls)
    lens = [len(d) for _, d, _, _ in calls]
    in_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    d_in = _to_device(b"".join(d for _, d, _, _ in calls))
    slots = [(cap + GUARD + 15) // 16 * 16 for _, _, cap, _ in calls]
    out_off = np.concatenate([[0], np.cumsum(slots)]).astype(np.int64)
    out = torch.full((int(out_off[-1]),), PAT, dtype=torch.uint8, device="cuda")
    res = torch.full((n, 2), -7, dtype=torch.int32, device="cuda")
    ws = torch.empty(max(cs.api.lib().csnappy_stream_decompress_workspace(lens[i], calls[i][2]) for i in range(n)),
                     dtype=torch.uint8, device="cuda")
    for i, (_, _, cap, _) in enumerate(calls):
        cs.api.stream_decompress(d_in[int(in_off[i]):], lens[i], cap, out=out[int(out_off[i]):], workspace=ws,
                                 result=res[i])
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    got = res.cpu().numpy()
    bad = []
    for i, (name, _, cap, (rc, _, exp)) in enumerate(calls):
        out_len, status = int(got[i, 0]), int(got[i, 1])
        slot = o[out_off[i]:out_off[i + 1]]
        if status != rc:
            bad.append((name, "status", status, rc))
        elif rc == 0 and (out_len != len(exp) or slot[:out_len].tobytes() != exp):
            bad.append((name, "output", out_len, len(exp)))
        elif rc != 0 and out_len != 0:
            bad.append((name, "out_len on error", out_len))
        if (slot[cap:] != PAT).any():
            bad.append((name, "wrote at or past cap", cap + int(np.nonzero(slot[cap:] != PAT)[0][0])))
    assert not bad, (len(bad), bad[:8])
    return n


def _shifted_calls(pairs):
    return [(f"{c.name} +{k}", C.ZERO_LIT * k + c.data, c.cap, c.expect()) for c, k in pairs]


def test_stream_decoder_shifted_invalid_cases(cs, plan):
    assert _stream_calls(cs, _shifted_calls(plan["invalid"])) == 6141


def test_stream_decoder_shifted_edge_streams(cs, plan):
    _stream_calls(cs, _shifted_calls(plan["edges"]))


def test_stream_decoder_shifted_copy_matrix(cs, plan):
    _stream_calls(cs, _shifted_calls(plan["copy_matrix"]))


def test_stream_decoder_chunk_cases(cs):
    _stream_calls(cs, [(c.name, c.data, c.cap, c.expect()) for c in C.chunk_cases(301)])


@pytest.mark.parametrize("stream_min", [0, -1], ids=["parallel", "serial"])
def test_dropin_long_branch_shifted(cs, plan, stream_min):
    """csnappy_decompress_noheader takes its long-stream branch above 64 KiB of input: the shifted cases with at least
    13 108 zero-length literals in front (a whole number of chunks more, so the phase stays)."""
    rng = np.random.default_rng(9)
    pairs = [p for part in ("invalid", "edges", "copy_matrix") for p in plan[part]]
    sample = [pairs[i] for i in rng.choice(len(pairs), 300, replace=False)]
    cs.set_tuning("stream_decode_min", stream_min)
    try:
        for c, k in sample:
            k += C.CHUNK * max(0, -(-(13108 - k) // C.CHUNK))
            data = C.ZERO_LIT * k + c.data
            assert len(data) > 65536
            rc, _, exp = c.expect()
            got_rc, got = cs.csnappy_decompress_noheader(data, c.cap)  # asserts *dst_len untouched on error
            assert got_rc == rc, (c.name, k, got_rc, rc)
            if rc == 0:
                assert got == exp, (c.name, k)
    finally:
        cs.set_tuning("stream_decode_min", 0)


# ---- capacities of 2^31 and above ---------------------------------------------------------------------------
def _result(res):
    """(status, out_len) of a stream decoder call; out_len read as the uint32 it is."""
    out_len, status = res.cpu().tolist()
    return status, out_len & 0xFFFFFFFF


def _guard_ok(out, at):
    return bool((out[at:at + GUARD] == PAT).all())


# (decompress_stage_input): global path; staged, where the 32 KiB out area sends the block to the global path; lanes
@pytest.mark.parametrize("stage", [3, 1, 4])
def test_big_capacity_literals_batch(cs, stage):
    cases = C.big_literal_cases(7)
    stride = (S.NO_CAP + GUARD + 15) // 16 * 16
    big_stride = (BIG + GUARD + 15) // 16 * 16
    out = torch.full((max(stride, 3 * big_stride) + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    cs.set_tuning("decompress_stage_input", stage)
    try:
        for c in cases:
            rc, _, _ = c.expect()
            d_in = _to_device(c.data)
            d_len = torch.tensor([len(c.data)], dtype=torch.int32, device="cuda")
            out[c.cap:c.cap + GUARD].fill_(PAT)
            _, out_len, status = cs.batch_decompress(d_in, d_len, 1, c.cap, out=out, out_stride=stride)
            torch.cuda.synchronize()
            assert (int(status[0]), int(out_len[0])) == (rc, 0), (c.name, int(status[0]), rc)
            assert _guard_ok(out, c.cap), c.name
        # per-block capacities: [p + 100, 2^31 + 2^20, a small valid block], the stride from the largest
        small = S.Case(S.random_stream(77, 3000), name="small valid block")
        for j in range(0, len(cases), 3):
            blocks = [cases[j], S.Case(cases[j].s, cap=BIG), small]
            caps = [b.cap for b in blocks]
            datas = [b.data for b in blocks]
            offs = np.concatenate([[0], np.cumsum([len(d) for d in datas])[:-1]]).astype(np.int64)
            d_in = _to_device(b"".join(datas))
            d_len = torch.tensor([len(d) for d in datas], dtype=torch.int32, device="cuda")
            d_caps = torch.from_numpy(np.array(caps, dtype=np.uint32).view(np.int32)).cuda()
            for i, cap in enumerate(caps):
                out[i * big_stride + cap:i * big_stride + cap + GUARD].fill_(PAT)
            _, out_len, status = cs.batch_decompress(d_in, d_len, 3, 0, in_off=torch.from_numpy(offs).cuda(), out=out,
                                                     out_stride=big_stride, out_caps=d_caps)
            torch.cuda.synchronize()
            for i, b in enumerate(blocks):
                rc, _, exp = b.expect()
                assert int(status[i]) == rc, (b.name, caps[i], int(status[i]), rc)
                assert int(out_len[i]) == (len(exp) if rc == 0 else 0), b.name
                assert _guard_ok(out, i * big_stride + caps[i]), (b.name, caps[i])
            got = out[2 * big_stride:2 * big_stride + len(small.expect()[2])].cpu().numpy().tobytes()
            assert got == small.expect()[2]
    finally:
        cs.set_tuning("decompress_stage_input", 0)
        del out
        torch.cuda.empty_cache()


def test_big_capacity_literals_stream_decoder(cs):
    """The stream decoder at a capacity of 2^31 + 2^20 (its workspace holds 4 bytes per capacity byte)."""
    cases = [S.Case(c.s, cap=BIG, name=c.name) for c in C.big_literal_cases(7) if c.cap == BIG]
    assert [c.expect()[0] for c in cases] == [S.E_DATA_MALFORMED, S.E_OUTPUT_OVERRUN, S.E_DATA_MALFORMED]
    out = torch.full((BIG + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    ws = torch.empty(max(cs.api.lib().csnappy_stream_decompress_workspace(len(c.data), BIG) for c in cases),
                     dtype=torch.uint8, device="cuda")
    try:
        for c in cases:
            _, res = cs.api.stream_decompress(_to_device(c.data), len(c.data), BIG, out=out, workspace=ws)
            torch.cuda.synchronize()
            assert _result(res) == (c.expect()[0], 0), c.name
            assert _guard_ok(out, BIG), c.name
    finally:
        del out, ws
        torch.cuda.empty_cache()


def test_stream_decoder_output_above_2_gib(cs):
    """2^31 + 2^20 bytes through the stream decoder: a 4 KiB literal, an offset-1 run, copy-4 tags whose offsets exceed
    2^31, a literal.  The run is a back-reference chain 2^31 deep for resolve_kernel.  The expected output is built
    on the device, so that 2 GiB never crosses to the host.  Capacity exactly the output: 0; one byte less: -3; a
    last copy-4 with an offset one past the output: -5."""
    r = C.RunStream(5, BIG)
    assert r.produced > BIG and all(o - x > 1 << 31 for o, x, _ in r.copies)
    bad = r.data + r.bad_offset_tail()
    d_in = _to_device(bad)
    head = torch.frombuffer(bytearray(r.head), dtype=torch.uint8).cuda()
    exp = torch.empty(r.produced, dtype=torch.uint8, device="cuda")
    exp[:C.CHUNK] = head
    exp[C.CHUNK:r.run_end].fill_(r.head[-1])
    for o, x, n in r.copies:
        exp[o:o + n] = head[x:x + n]
    exp[r.produced - len(r.tail):] = torch.frombuffer(bytearray(r.tail), dtype=torch.uint8).cuda()
    runs = [(len(r.data), r.produced, 0), (len(r.data), r.produced - 1, S.E_OUTPUT_OVERRUN),
            (len(bad), r.produced + 8, S.E_DATA_MALFORMED)]
    ws = torch.empty(max(cs.api.lib().csnappy_stream_decompress_workspace(n, cap) for n, cap, _ in runs),
                     dtype=torch.uint8, device="cuda")
    out = torch.empty(r.produced + 8 + GUARD, dtype=torch.uint8, device="cuda")
    try:
        for n, cap, rc in runs:
            out.fill_(PAT)
            _, res = cs.api.stream_decompress(d_in, n, cap, out=out, workspace=ws)
            torch.cuda.synchronize()
            assert _result(res) == (rc, r.produced if rc == 0 else 0), (cap, _result(res))
            assert _guard_ok(out, cap), cap
            if rc == 0:
                assert torch.equal(out[:r.produced], exp)
    finally:
        del out, ws, exp
        torch.cuda.empty_cache()


def test_stream_decoder_saturated_output_offset(cs):
    """A copy that does not fit, then more than 2^32 bytes of copies: the running output offset saturates, the
    earlier failure decides (-3) and nothing at or past the capacity changes."""
    data, cap = C.saturating_stream(2)
    out = torch.full((cap + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    ws = torch.empty(cs.api.lib().csnappy_stream_decompress_workspace(len(data), cap), dtype=torch.uint8,
                     device="cuda")
    try:
        _, res = cs.api.stream_decompress(_to_device(data), len(data), cap, out=out, workspace=ws)
        torch.cuda.synchronize()
        assert _result(res) == (S.E_OUTPUT_OVERRUN, 0)
        assert _guard_ok(out, cap)
    finally:
        del out, ws
        torch.cuda.empty_cache()
