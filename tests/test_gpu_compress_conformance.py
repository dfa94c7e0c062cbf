"""Every GPU compress form against the oracle, on blocks built to drive the kernel's rarely taken paths.

tests/compress_cases.py plants hash-slot sharing (pairs at every distance, three and four words on one slot,
A-B-A, true repeats plus a collision, interleaved and nested pairs) at the block start, behind copies, after
in-window copies and in strided windows; short and chained copies; the scan end; match, literal and copy lengths
at the kernel's step and header boundaries; offsets at the copy-1 limit; 31..65 copies per block.  Here those
blocks go through the lane groups 32 / 16 / 8, the staged and the global-memory 32-lane forms, strided and
packed (odd-aligned, through in_off) layouts with uniform and per-block lengths, BATCH_SHRINK_TABLE, and the
whole-buffer calls.  Bytes and out_len must equal the oracle's, and nothing past out_len of a slot, or past the
last slot, may change: the emitters write exactly the bytes they emit.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import compress_cases as CC  # noqa: E402
import oracle  # noqa: E402

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAT = 0xA5
GUARD = 256
WMS = (9, 13, 15, 16)


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.fixture(scope="module")
def chk():
    return oracle.best()


@pytest.fixture(scope="module")
def sets():
    """wm -> [(name, blocks, uniform length or None)]: the 4 KiB and 32 KiB blocks, and a ragged mix with the short
    blocks and final-literal cases."""
    short = [c.data for c in CC.size_cases()]
    out = {}
    for wm in WMS:
        cor = CC.corpus(wm)
        b4 = [c.data for c in cor if len(c.data) == 4096]
        b32 = [c.data for c in cor if len(c.data) == 32768]
        mixed = short + b4[::3] + [b[: len(b) - k] for k, b in enumerate(b32[:4])] + [b4[0][:4095], b4[1][:17]]
        out[wm] = [("4k", b4, 4096), ("32k", b32, 32768), ("mixed", mixed, None)]
    return out


def _layout(blocks, layout, uniform):
    lens = np.array([len(b) for b in blocks], dtype=np.int32)
    if layout == "stride":
        stride = uniform if uniform else max(lens)
        host = np.zeros((len(blocks), stride), dtype=np.uint8)
        for i, b in enumerate(blocks):
            host[i, : len(b)] = np.frombuffer(b, dtype=np.uint8)
        return torch.from_numpy(host.reshape(-1)).cuda(), lens, dict(in_stride=stride)
    # back to back from an odd address: every block at its own alignment mod 16
    offs = np.zeros(len(blocks), dtype=np.int64)
    pos = 1
    for i, b in enumerate(blocks):
        offs[i] = pos
        pos += len(b)
    host = np.zeros(pos + 64, dtype=np.uint8)
    for i, b in enumerate(blocks):
        host[offs[i]: offs[i] + len(b)] = np.frombuffer(b, dtype=np.uint8)
    return torch.from_numpy(host).cuda(), lens, dict(in_off=torch.from_numpy(offs).cuda())


def _compress_and_check(cs, chk, blocks, wm, layout, uniform, flags=0, wms=None):
    B = len(blocks)
    block_len = uniform or max(len(b) for b in blocks)
    stride = cs.api.out_stride_for(block_len)
    d_in, lens, kw = _layout(blocks, layout, uniform)
    if not uniform or layout == "packed":
        kw["in_len"] = torch.from_numpy(lens).cuda()
    out = torch.full((B * stride + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    out_len = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    cs.batch_compress_fragments(d_in, block_len, B, wm, out=out, out_len=out_len, out_stride=stride, flags=flags, **kw)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    assert (o[B * stride:] == PAT).all(), "wrote past the last slot"
    got_len = out_len.cpu().numpy()
    bad = []
    for i, b in enumerate(blocks):
        w = wms[i] if wms else wm
        exp = chk.compress_fragment(b, w)
        slot = o[i * stride:(i + 1) * stride]
        if got_len[i] != len(exp) or slot[: len(exp)].tobytes() != exp:
            bad.append((i, len(b), w, int(got_len[i]), len(exp)))
        elif not (slot[len(exp):] == PAT).all():
            bad.append((i, len(b), w, "wrote past out_len at", len(exp) + int(np.flatnonzero(slot[len(exp):] != PAT)[0])))
        if len(bad) >= 8:
            break
    assert not bad, bad


# (compress_lanes, compress_stage_input): staged 32 / 16 / 8 lanes, 32 lanes from global memory, forced staging
CONFIGS = [(32, 0), (16, 0), (8, 0), (32, 2), (32, 1)]


@pytest.mark.parametrize("layout", ["stride", "packed"])
@pytest.mark.parametrize("lanes,stage", CONFIGS)
def test_batch_compress_conformance(cs, chk, sets, lanes, stage, layout):
    cs.set_tuning("compress_lanes", lanes)
    cs.set_tuning("compress_stage_input", stage)
    try:
        for wm in WMS:
            for name, blocks, n in sets[wm]:
                _compress_and_check(cs, chk, blocks, wm, layout, n if layout == "stride" else None)
                if layout == "stride" and n:
                    # the same blocks with per-block lengths (uniform)
                    _compress_and_check(cs, chk, blocks, wm, "stride", None)
    finally:
        cs.set_tuning("compress_lanes", 0)
        cs.set_tuning("compress_stage_input", 0)


@pytest.mark.parametrize("lanes,stage", [(32, 0), (16, 0), (32, 2)])
def test_batch_compress_shrink_table(cs, chk, lanes, stage):
    """BATCH_SHRINK_TABLE at wm 9-16: lengths 2^k - 1, 2^k, 2^k + 1 for k = 8..15 take csnappy_compress's table size
    for a short last chunk (oracle chunk_wm)."""
    src = b"".join(c.data for c in CC.corpus(13) if len(c.data) == 4096)
    lens = [x for k in range(8, 16) for x in ((1 << k) - 1, 1 << k, (1 << k) + 1) if x <= 32768]
    cs.set_tuning("compress_lanes", lanes)
    cs.set_tuning("compress_stage_input", stage)
    try:
        for wm in range(9, 17):
            blocks = [src[37 * i: 37 * i + n] for i, n in enumerate(lens)]
            wms = [oracle.port().chunk_wm(n, wm) for n in lens]
            _compress_and_check(cs, chk, blocks, wm, "packed", None, flags=cs.api.BATCH_SHRINK_TABLE, wms=wms)
    finally:
        cs.set_tuning("compress_lanes", 0)
        cs.set_tuning("compress_stage_input", 0)


def test_whole_buffers(cs, chk):
    """Concatenations of generated blocks over several 32 KiB fragments with a short last chunk, through the drop-in
    csnappy_compress and through csnappy_batch_compress."""
    src = b"".join(c.data for wm in (9, 16) for c in CC.corpus(wm))
    bufs = [src[:70001], src[5:5 + 32768 + 15], src[100:100 + 65536 + 4097], src[7:7 + 3 * 32768 + 1], src[:32769],
            src[11:11 + 40000]]
    offs, pos = [], 0
    for b in bufs:
        offs.append(pos)
        pos += len(b) + 5
    host = np.zeros(pos + 16, dtype=np.uint8)
    for o, b in zip(offs, bufs):
        host[o:o + len(b)] = np.frombuffer(b, dtype=np.uint8)
    d_in = torch.from_numpy(host).cuda()
    for wm in (9, 13, 15, 16):
        exp = [chk.compress(b, wm) for b in bufs]
        for b, e in zip(bufs[:3], exp):
            assert cs.csnappy_compress(b, wm) == e, (len(b), wm)
        out, out_len, stride = cs.api.batch_compress(d_in, offs, [len(b) for b in bufs], wm)
        o, ol = out.cpu().numpy(), out_len.cpu().numpy()
        for i, e in enumerate(exp):
            assert o[i * stride: i * stride + ol[i]].tobytes() == e, (i, len(bufs[i]), wm)
