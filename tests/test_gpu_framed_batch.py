"""Many framed streams in one device call (csnappy_framed_batch_*) against the restatement (tests/framed.py) and against
N single calls: writer bytes at every wm and layout, reader results on every hostile stream in one batch (reversed and
shuffled too, through every decoder routing), the declared-length call, launch counts independent of the stream count,
refused arguments, and a batch above 1 GiB.  Every output buffer is pre-filled with 0xA5 and the bytes between and
behind the slots must survive."""
from __future__ import annotations

import numpy as np
import pytest

import framed as F
import framed_batch as FB
import oracle
import streams

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from csnappy_b200 import api  # noqa: E402
from csnappy_b200._lib import lib  # noqa: E402

FILL = 0xA5
GUARD = 4096


def _u64(xs):
    return np.ascontiguousarray(np.asarray(xs, dtype=np.uint64))


def _dev(b: bytes):
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


def batch_compress(bufs, wm, *, gaps_seed=None, seed=0):
    """The batch writer with inputs at odd offsets; output slots back to back (gaps_seed None: NULL h_out_off) or with
    gaps.  Checks the guard bytes and returns the streams."""
    src, offs = FB.packed(bufs, seed)
    d = _dev(src)
    m = [F.max_length(len(b)) for b in bufs]
    if gaps_seed is None:
        out_off, end = list(np.concatenate(([0], np.cumsum(m)[:-1])).astype(np.int64)) if bufs else [], sum(m)
    else:
        out_off, end = FB.slots_with_gaps(m, gaps_seed)
    out = torch.full((end + GUARD,), FILL, dtype=torch.uint8, device="cuda")
    o, h_out, olen = api.framed_batch_compress_device(d, offs, [len(b) for b in bufs], wm,
                                                      out_off=None if gaps_seed is None else out_off, out=out)
    torch.cuda.synchronize()
    assert [int(x) for x in h_out] == [int(x) for x in out_off]
    raw = bytes(out.cpu().numpy())
    ol = olen.cpu().tolist()[: len(bufs)]
    got = [raw[int(s):int(s) + n] for s, n in zip(out_off, ol)]
    assert not FB.untouched_outside(raw, [(int(s), int(s) + n) for s, n in zip(out_off, ol)]), "bytes outside the slots"
    return got


def single_compress(bufs, wm):
    L = lib()
    s = torch.cuda.current_stream().cuda_stream
    longest = max([len(b) for b in bufs] + [1])
    d = torch.empty(longest + 8, dtype=torch.uint8, device="cuda")
    out = torch.empty(F.max_length(longest), dtype=torch.uint8, device="cuda")
    olen = torch.empty(1, dtype=torch.int64, device="cuda")
    ws = torch.empty(L.csnappy_framed_compress_workspace(longest), dtype=torch.uint8, device="cuda")
    res = []
    for b in bufs:
        if b:
            d[:len(b)] = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
        assert L.csnappy_framed_compress(d.data_ptr(), len(b), out.data_ptr(), out.numel(), olen.data_ptr(), wm,
                                         ws.data_ptr(), ws.numel(), s) == 0
        res.append(bytes(out[: int(olen.item())].cpu().numpy()))
    return res


@pytest.fixture(scope="module")
def edges():
    port = oracle.port()
    return [F.edge_chunk(n, 16, d, port=port) for n in (F.CHUNK, 4096) for d in (-1, 0, 1)]


# ---------------------------------------------------------------------------------------------------- writer
@pytest.mark.parametrize("wm", range(9, 17))
def test_writer_matches_restatement(wm, edges):
    port = oracle.port()
    rng = np.random.default_rng(wm)
    bufs = [F.mixed_bytes(n + 1, n, scale=9000) for n in F.LENGTHS if n < 2**20 or wm in (9, 16)]
    bufs = bufs[:5] + [e for e in edges if e is not None] + bufs[5:]
    bufs += [F.mixed_bytes(100 + i, int(rng.integers(0, 300000)), scale=int(rng.integers(64, 70000))) for i in range(12)]
    exp = [F.write_framed(b, wm, port) for b in bufs]
    assert batch_compress(bufs, wm, seed=wm) == exp
    assert batch_compress(bufs, wm, gaps_seed=wm, seed=wm + 1) == exp


def test_writer_matches_single_calls_small_cases():
    for bufs in ([b""] * 7, [F.mixed_bytes(3, 200001, scale=5000)], [b"", b"x", b""],
                 [F.mixed_bytes(i, n, scale=300) for i, n in enumerate((0, 1, 65536, 65537, 32768, 32769, 0, 7))]):
        for wm in (9, 13, 16):
            assert batch_compress(bufs, wm) == single_compress(bufs, wm)


def test_writer_100000_tiny_streams():
    rng = np.random.default_rng(5)
    lens = rng.integers(1, 101, 100000)
    pool = F.mixed_bytes(6, 200000, scale=50)
    starts = rng.integers(0, len(pool) - 100, 100000)
    bufs = [pool[s:s + n] for s, n in zip(starts, lens)]
    got = batch_compress(bufs, 12, gaps_seed=3)
    assert got == single_compress(bufs, 12)


def test_writer_more_than_65536_chunks():
    """1100 streams of 60 to 64 chunks (about 4.5 GiB, more than 65536 chunks), every slot compared on the device with
    a single call, and the guard bytes between and behind the slots checked."""
    g = torch.Generator(device="cuda").manual_seed(9)
    rng = np.random.default_rng(9)
    lens = [int(x) for x in rng.integers(60 * F.CHUNK, 64 * F.CHUNK + 1, 1100)]
    offs = np.concatenate(([3], 3 + np.cumsum(lens)[:-1])).astype(np.int64)
    total = int(offs[-1]) + lens[-1] + 8
    d = torch.randint(97, 105, (total,), dtype=torch.uint8, device="cuda", generator=g)
    d[: total // 4] = torch.randint(0, 256, (total // 4,), dtype=torch.uint8, device="cuda", generator=g)
    assert sum(-(-n // F.CHUNK) for n in lens) > 65536
    slot_off, end = FB.slots_with_gaps([F.max_length(n) for n in lens], 9)
    out = torch.full((end + GUARD,), FILL, dtype=torch.uint8, device="cuda")
    _, _, olen = api.framed_batch_compress_device(d, offs, lens, 14, out_off=slot_off, out=out)
    ol = olen.cpu().tolist()
    one = torch.empty(F.max_length(max(lens)), dtype=torch.uint8, device="cuda")
    written = torch.zeros(out.numel(), dtype=torch.bool, device="cuda")
    for i in range(len(lens)):
        o, n1 = api.framed_compress_device(d[int(offs[i]):], lens[i], 14, out=one)
        n1 = int(n1.item())
        assert ol[i] == n1, i
        assert torch.equal(out[slot_off[i]:slot_off[i] + n1], o[:n1]), i
        written[slot_off[i]:slot_off[i] + n1] = True
    assert bool((out[~written] == FILL).all()), "bytes outside the slots"


# ---------------------------------------------------------------------------------------------------- reader
@pytest.fixture(scope="module")
def hostile():
    return F.hostile_streams(11, 16, stream_cases=streams.boundary_streams(7)[::3] + streams.copy_matrix(7, phases=(0,))[::60])


SENTINEL = 0x5EED5EED5EED


def batch_decompress(items, seed=0, place=None):
    """items: [(stream, cap)] in one batch at odd source offsets, output slots with gaps; guard bytes checked.
    place: the order in which the streams lie in the source buffer (default: stream order).
    -> [(rc, out_len, failed_offset or None, prefix)]; the sentinel must survive on streams that succeed."""
    bufs = [s for s, _ in items]
    caps = [c for _, c in items]
    place = list(range(len(bufs))) if place is None else list(place)
    src, at = FB.packed([bufs[i] for i in place], seed)
    offs = [0] * len(bufs)
    for k, i in enumerate(place):
        offs[i] = at[k]
    dst_off, end = FB.slots_with_gaps(caps, seed + 1)
    dst = torch.full((end + GUARD,), FILL, dtype=torch.uint8, device="cuda")
    fo = torch.full((len(items),), SENTINEL, dtype=torch.int64, device="cuda")
    _, _, res = api.framed_batch_decompress_device(_dev(src), offs, [len(b) for b in bufs], caps, dst_off=dst_off, dst=dst,
                                                  failed_offset=fo)
    torch.cuda.synchronize()
    raw = bytes(dst.cpu().numpy())
    r = res.cpu().tolist()
    assert not FB.untouched_outside(raw, [(o, o + c) for o, c in zip(dst_off, caps)]), "bytes outside the capacities"
    out = []
    for i in range(len(items)):
        n, rc, bad = r[0][i], r[1][i], r[2][i]
        if rc == 0:
            assert bad == SENTINEL, i
        out.append((rc, n, bad if rc else None, raw[dst_off[i]:dst_off[i] + n]))
    return out


def _expect(items):
    return [F.read_framed(s, c) for s, c in items]


def _compare(got, exp, names):
    for g, e, name in zip(got, exp, names):
        assert g[:3] == e.key(), name
        assert g[3] == e.data, name


def test_reader_on_every_hostile_stream_in_one_batch(hostile):
    items = [(h.stream, h.cap) for h in hostile]
    exp = _expect(items)
    names = [h.cls for h in hostile]
    _compare(batch_decompress(items, 1), exp, names)
    _compare(batch_decompress(items[::-1], 2), exp[::-1], names[::-1])
    perm = np.random.default_rng(3).permutation(len(items))
    _compare(batch_decompress([items[i] for i in perm], 3), [exp[i] for i in perm], [names[i] for i in perm])
    # streams lying in the source buffer in another order than their stream index
    _compare(batch_decompress(items, 4, place=perm), exp, names)


@pytest.mark.parametrize("stage", [1, 2, 3, 4])
def test_reader_every_decoder_path(hostile, stage):
    pick = [h for h in hostile if h.cls in ("foreign_chunking", "valid", "two_failures_decode_crc", "concatenated",
                                            "two_failures_crc_decode", "varint_short", "capacity_short")]
    pick += [h for h in hostile if h.cls == "tag_forms"][::4]
    items = [(h.stream, h.cap) for h in pick]
    api.set_tuning("decompress_stage_input", stage)
    try:
        _compare(batch_decompress(items, stage), _expect(items), [h.cls for h in pick])
    finally:
        api.set_tuning("decompress_stage_input", 0)


def test_bytes_list_round_trip():
    bufs = [F.mixed_bytes(i, n, scale=3000) for i, n in enumerate((0, 1, 100, 65536, 65537, 300000, 0))]
    zs = api.framed_batch_compress(bufs, 13)
    assert zs == [F.write_framed(b, 13) for b in bufs]
    assert api.framed_batch_decompress(zs) == [(0, b, None) for b in bufs]
    assert api.framed_batch_compress([]) == [] and api.framed_batch_decompress([]) == []


# ---------------------------------------------------------------------------------------------------- length call
def test_decompressed_length(hostile):
    valid = [F.write_framed(F.mixed_bytes(i, n, scale=2000), 16) for i, n in enumerate((0, 1, 65536, 65537, 200000))]
    bufs = [h.stream for h in hostile] + valid
    src, offs = FB.packed(bufs, 4)
    length, status = api.framed_batch_decompressed_length_device(_dev(src), offs, [len(b) for b in bufs])
    torch.cuda.synchronize()
    got = list(zip(length.cpu().tolist(), status.cpu().tolist()))
    exp = [FB.declared_length(b) for b in bufs]
    assert got == exp
    # decoding with that capacity never runs out of room
    res = batch_decompress([(b, n) for b, (n, _) in zip(bufs, exp)], 5)
    assert all(r[0] != F.E_OUTPUT_INSUF for r in res)
    assert api.framed_batch_decompress(valid) == [(0, F.read_framed(v, 1 << 30).data, None) for v in valid]


# ---------------------------------------------------------------------------------------------------- launches
def test_launch_count_does_not_grow_with_the_batch():
    data = F.mixed_bytes(2, 70000, scale=3000)  # a compressed and a stored chunk
    z = F.write_framed(data, 13)

    def launches(fn):
        torch.cuda.synchronize()
        k = api.kernel_launches()
        fn()
        torch.cuda.synchronize()
        return api.kernel_launches() - k

    counts = {}
    for n in (1, 10000):
        d, offs, lens = api._stage([data] * n)
        dz, zoffs, zlens = api._stage([z] * n)
        counts[n] = (launches(lambda: api.framed_batch_compress_device(d, offs, lens, 13)),
                     launches(lambda: api.framed_batch_decompress_device(dz, zoffs, zlens, [len(data)] * n)),
                     launches(lambda: api.framed_batch_decompressed_length_device(dz, zoffs, zlens)))
    assert counts[1] == counts[10000], counts
    assert all(c > 0 for c in counts[1])


# ---------------------------------------------------------------------------------------------------- refused
def test_refused_arguments():
    L = lib()
    BAD = api.CSNAPPY_E_BAD_ARG
    buf = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    p, ws = buf.data_ptr(), buf.data_ptr() + (1 << 19)
    s = torch.cuda.current_stream().cuda_stream
    lens, offs = _u64([1000, 0, 3000]), _u64([0, 1000, 1001])
    L_, O_ = lens.ctypes.data, offs.ctypes.data
    cap = sum(F.max_length(int(n)) for n in lens)
    wsc = L.csnappy_framed_batch_compress_workspace(L_, 3)
    outl = p + 200000
    good = [p, O_, L_, 3, p + 8192, None, cap, outl, 16, ws, wsc, s]
    assert L.csnappy_framed_batch_compress(*good) == 0
    torch.cuda.synchronize()
    out_off = _u64([0, 2000, 4000])
    for k, v in ((8, 8), (8, 17), (10, wsc - 1), (6, cap - 1), (0, None), (1, None), (2, None), (4, None), (7, None),
                 (9, None)):
        args = list(good)
        args[k] = v
        assert L.csnappy_framed_batch_compress(*args) == BAD, (k, v)
    args = list(good)
    args[5], args[6] = out_off.ctypes.data, 4000 + F.max_length(3000) - 1  # the last slot ends one byte past
    assert L.csnappy_framed_batch_compress(*args) == BAD
    args[6] += 1
    assert L.csnappy_framed_batch_compress(*args) == 0
    huge = _u64([(2**32 - 2) * 32768 + 1])
    assert L.csnappy_framed_batch_compress_workspace(huge.ctypes.data, 1) == 2**64 - 1
    assert L.csnappy_framed_batch_compress(p, O_, huge.ctypes.data, 1, p, None, 2**63, outl, 16, ws, 2**63, s) == BAD
    many = _u64([2**31 * 32768] * 2 + [32768])  # 2^32 + 1 fragments in all
    many_off = _u64([0, 0, 0])
    assert L.csnappy_framed_batch_compress(p, many_off.ctypes.data, many.ctypes.data, 3, p, None, 2**63, outl, 16, ws,
                                           2**63, s) == BAD
    assert L.csnappy_framed_batch_compress(p, O_, L_, 0, None, None, 0, None, 16, None, 0, s) == 0
    # reader
    caps = _u64([100, 100, 100])
    dst_off = _u64([0, 100, 200])
    wsd = L.csnappy_framed_batch_decompress_workspace(L_, 3)
    good = [p, O_, L_, 3, p + 8192, dst_off.ctypes.data, caps.ctypes.data, outl, outl + 64, outl + 128, ws, wsd, s]
    assert L.csnappy_framed_batch_decompress(*good) == 0
    for k in (0, 1, 2, 4, 5, 6, 7, 8, 10):
        args = list(good)
        args[k] = None
        assert L.csnappy_framed_batch_decompress(*args) == BAD, k
    args = list(good)
    args[11] = wsd - 1
    assert L.csnappy_framed_batch_decompress(*args) == BAD
    big = _u64([2**35 + 1])
    assert L.csnappy_framed_batch_decompress_workspace(big.ctypes.data, 1) == 2**64 - 1
    args = list(good)
    args[2], args[3] = big.ctypes.data, 1
    assert L.csnappy_framed_batch_decompress(*args) == BAD
    entries = _u64([2**35 - 16] * 2)  # 2 * (2^32 - 1) table entries
    args = list(good)
    args[2], args[3] = entries.ctypes.data, 2
    assert L.csnappy_framed_batch_decompress(*args) == BAD
    assert L.csnappy_framed_batch_decompressed_length(p, O_, big.ctypes.data, 1, outl, outl + 64, s) == BAD
    for k in (1, 2, 4, 5):
        args = [p, O_, L_, 3, outl, outl + 64, s]
        args[k] = None
        assert L.csnappy_framed_batch_decompressed_length(*args) == BAD, k
    assert L.csnappy_framed_batch_decompress(None, None, None, 0, None, None, None, None, None, None, None, 0, s) == 0
    assert L.csnappy_framed_batch_decompressed_length(None, None, None, 0, None, None, s) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- large
def test_large_batch_round_trip_and_one_flipped_bit():
    """Thousands of streams of mixed sizes up to 256 KiB, more than 1 GiB in all; one flipped bit in one stream's
    stored chunk fails only that stream, with -102 at that chunk and the chunks before it intact."""
    rng = np.random.default_rng(21)
    lens = [int(x) for x in rng.choice([int(rng.integers(0, 4096)), 4096, 65536, 100000, 262144], 6000)]
    lens = [int(rng.integers(0, 262145)) if i % 3 == 0 else n for i, n in enumerate(lens)]
    while sum(lens) <= (1 << 30):
        lens.append(262144)
    offs = np.concatenate(([0], np.cumsum(lens)[:-1])).astype(np.int64)
    total = sum(lens)
    g = torch.Generator(device="cuda").manual_seed(4)
    d = torch.randint(97, 101, (total + 8,), dtype=torch.uint8, device="cuda", generator=g)
    d[: total // 3] = torch.randint(0, 256, (total // 3,), dtype=torch.uint8, device="cuda", generator=g)
    z, z_off, zlen = api.framed_batch_compress_device(d, offs, lens, 16)
    zl = zlen.cpu().tolist()[: len(lens)]
    dst, dst_off, res = api.framed_batch_decompress_device(z, z_off, zl, lens)
    torch.cuda.synchronize()
    r = res.cpu().tolist()
    assert r[1][: len(lens)] == [0] * len(lens) and r[0][: len(lens)] == lens
    assert torch.equal(dst[:total], d[:total])
    # stream j: random bytes at the front of the input, so its chunks are stored; flip a bit in its third chunk
    j = next(i for i in range(len(lens)) if lens[i] > 3 * F.CHUNK and offs[i] + lens[i] < total // 3)
    zs = z[int(z_off[j]):int(z_off[j]) + zl[j]].cpu().numpy()
    pos = 10
    for _ in range(2):
        pos += 4 + int(zs[pos + 1]) + (int(zs[pos + 2]) << 8) + (int(zs[pos + 3]) << 16)
    assert zs[pos] == 1
    z[int(z_off[j]) + pos + 100] ^= 4
    dst.fill_(0)
    dst, _, res = api.framed_batch_decompress_device(z, z_off, zl, lens, dst=dst)
    torch.cuda.synchronize()
    r = res.cpu().tolist()
    for i in range(len(lens)):
        want = (2 * F.CHUNK, F.E_CHECKSUM, pos) if i == j else (lens[i], 0, -1)
        assert (r[0][i], r[1][i], r[2][i]) == want, i
    o = int(dst_off[j])
    assert torch.equal(dst[o:o + 2 * F.CHUNK], d[int(offs[j]):int(offs[j]) + 2 * F.CHUNK])
    assert torch.equal(dst[:o], d[:o])
    assert torch.equal(dst[o + lens[j]:total], d[o + lens[j]:total])
