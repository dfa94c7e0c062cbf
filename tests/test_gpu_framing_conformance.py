"""The layer above the kernels against plain restatements: the page container writer and reader, csnappy_batch_compress
framing, csnappy_batch_pack, the drop-in csnappy_compress chunking and the strided host batch calls.

tests/containers.py restates the writer, the reader and the framing; tests/test_container_conformance.py checks those
against the oracle port and the generated inputs' coverage.  Here the same inputs go through the library:
  container  page sizes 1 ... 32768 (not multiples of 4 or 16 too, so every raw page source in gather_kernel is
             misaligned), pages whose compressed size is page + 1, page and page - 1 (the stored-block rule at
             equality), stored short last pages, last chunks of one page, chunk_mb 0 and 1, one device and device 0
             listed 1, 3 and 5 times (more workers than chunks), pinned, pageable and no_bounce caller memory, caller
             pointers at odd offsets; the reader on every hostile index of containers.hostile_containers, and under
             every decoder choice and lane group.
  framing    buffer lengths at every varint header length change up to 2^28, thousands of empty buffers, more than
             4096 fragments, the strided and uniform forms, refusal of short strides and workspaces.
  pack       n around the scan's 1024 threads and far above, odd strides and base offsets, offsets only.
  host calls chunk_mb 1 (1024-block chunks) with 4097 blocks, odd strides, ragged lengths, WITH_HEADER and RAW_IF_FULL,
             failures in later chunks, every slot with a 256-byte guard band behind its capacity.
Every output is pre-filled with a pattern: bytes a call does not own must stay as they were.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import containers as K  # noqa: E402
import oracle  # noqa: E402

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAT = 0xA5
GUARD = 256
PAGES = {1: 9, 3: 10, 17: 11, 64: 12, 1000: 13, 4095: 14, 4096: 13, 4097: 15, 16384: 16, 20000: 14, 32767: 15,
         32768: 16}


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.fixture(scope="module")
def chk():
    return oracle.best()


class knobs:
    """set_tuning for the duration of a block; every knob back to its default afterwards."""

    def __init__(self, cs, **kv):
        self.cs, self.kv = cs, kv

    def __enter__(self):
        for k, v in self.kv.items():
            self.cs.set_tuning(k, v)

    def __exit__(self, *exc):
        for k in self.kv:
            self.cs.set_tuning(k, 0)


def hostbuf(mem, n, off=0, fill=PAT):
    """n bytes of caller memory at offset `off` into a pattern-filled allocation with a guard band behind it.
    -> (keep-alive, whole numpy array, pointer of byte 0)."""
    t = torch.full((off + n + GUARD,), fill, dtype=torch.uint8)
    if mem == "pinned":
        t = t.pin_memory()
    a = t.numpy()
    return t, a, a.ctypes.data + off


def fill_host(mem, data: bytes, off=0):
    t, a, p = hostbuf(mem, len(data), off, fill=0x3C)
    a[off:off + len(data)] = np.frombuffer(data, dtype=np.uint8)
    return t, a, p


def dev_list(devices):
    if devices is None or devices == "single":
        return None, 0
    return (C.c_int * len(devices))(*devices), len(devices)


# ----------------------------------------------------------------------------------------------- container writer
# (chunk_mb, devices, caller memory, pointer offset); "single" = csnappy_bc_*_host, else the _multi call
VARIANTS = [(0, "single", "pinned", 0), (1, "single", "pageable", 1), (1, None, "no_bounce", 3), (0, [0], "pageable", 3),
            (1, [0, 0, 0], "pinned", 1), (1, [0] * 5, "pageable", 0), (0, [0, 0, 0], "no_bounce", 3),
            (0, [0] * 5, "pinned", 1)]


def bc_write(cs, data: bytes, page: int, wm: int, devices, mem, off):
    L = cs.api.lib()
    cap = cs.api.bc_max_container_length(len(data), page)
    keep_in, _, p_in = fill_host(mem, data, off)
    keep_out, a_out, p_out = hostbuf(mem, cap, (off * 5) % 4)
    o = (off * 5) % 4
    clen = C.c_uint64(0)
    if devices == "single":
        rc = L.csnappy_bc_compress_host(p_in, len(data), page, p_out, cap, C.byref(clen), wm)
    else:
        dv, nd = dev_list(devices)
        rc = L.csnappy_bc_compress_host_multi(p_in, len(data), page, p_out, cap, C.byref(clen), wm, dv, nd)
    assert rc == 0, cs.api.last_error()
    n = clen.value
    assert (a_out[:o] == PAT).all() and (a_out[o + n:] == PAT).all(), "container writer wrote past its length"
    del keep_in, keep_out
    return a_out[o:o + n].tobytes()


def bc_read(cs, cont: bytes, page: int, devices, mem, off, cap_bytes=None):
    """-> (rc, out_length, failed_page or None, output bytes [0, cap), whole output allocation ok behind cap)"""
    L = cs.api.lib()
    nr = int.from_bytes(cont[:4], "little") if len(cont) >= 4 else 0
    cap = nr * page if cap_bytes is None else cap_bytes
    cap = min(cap, 1 << 34)
    keep_in, _, p_in = fill_host(mem, cont, off)
    keep_out, a_out, p_out = hostbuf(mem, cap, 3 - off % 4)
    o = 3 - off % 4
    olen, bad = C.c_uint64(0), C.c_uint32(0xFFFFFFFF)
    if devices == "single":
        rc = L.csnappy_bc_decompress_host(p_in, len(cont), page, p_out, cap, C.byref(olen), C.byref(bad))
    else:
        dv, nd = dev_list(devices)
        rc = L.csnappy_bc_decompress_host_multi(p_in, len(cont), page, p_out, cap, C.byref(olen), C.byref(bad), dv, nd)
    assert rc not in (cs.api.CSNAPPY_E_DEVICE, cs.api.CSNAPPY_E_BAD_ARG), cs.api.last_error()
    assert (a_out[:o] == PAT).all() and (a_out[o + cap:] == PAT).all(), "container reader wrote outside its output"
    out = a_out[o:o + cap].copy()
    del keep_in, keep_out
    return rc, olen.value, (bad.value if rc != 0 and bad.value != 0xFFFFFFFF else None), out


def check_read(got, want: K.ReadResult, page, what, untouched_after_prefix=False):
    rc, olen, bad, out = got
    assert (rc, olen, bad) == want.key(), (what, want.key())
    for i, b in want.pages.items():
        assert out[i * page: i * page + len(b)].tobytes() == b, (what, "page", i)
    if untouched_after_prefix and want.rc not in (K.E_OUTPUT_INSUF, K.E_BAD_ARG):
        assert (out[want.prefix * page:] == PAT).all(), (what, "wrote a page past the decodable prefix")


@pytest.mark.parametrize("page", list(PAGES))
def test_container_writer_and_reader(cs, chk, page):
    wm = PAGES[page]
    tail = 1 + page % 31 if page > 31 else 0
    data, _ = K.container_input(page, wm, seed=17, tail=tail)
    inputs = [(data, VARIANTS)]
    for j, n in enumerate(K.edge_lengths(page)):
        inputs.append((K.mixed_bytes(1000 + j, n, scale=max(page, 64)), [VARIANTS[j % 8], VARIANTS[(j + 3) % 8]]))
    if page > 31:  # a stored short last page that is a Snappy literal: it decodes, one byte short
        inputs.append((data[: len(data) - tail] + K.short_tail(3, tail, snappy=True), VARIANTS[:2]))
    fewer_chunks = False
    for x, variants in inputs:
        ref = K.ref_container(chk, x, page, wm)
        nr = (len(x) + page - 1) // page
        want = K.read_container(ref, page, nr * page)
        for mb, devices, mem, off in variants:
            what = (page, len(x), mb, devices, mem, off)
            G = 1 if devices == "single" else (len(devices) if devices else cs.api.device_count())
            fewer_chunks |= -(-nr // K.chunk_pages(page, nr, G, mb)) < G
            with knobs(cs, chunk_mb=mb, no_bounce=int(mem == "no_bounce")):
                got = bc_write(cs, x, page, wm, devices, "pinned" if mem == "pinned" else "pageable", off)
                assert len(got) == len(ref) and got == ref, what
                check_read(bc_read(cs, ref, page, devices, "pinned" if mem == "pinned" else "pageable", off), want,
                           page, what)
    assert fewer_chunks  # some call had more workers than chunks


@pytest.mark.parametrize("page", [4096, 1000])
def test_container_reader_on_hostile_indexes(cs, chk, page):
    wm = PAGES[page]
    nr = 1100
    data = K.mixed_bytes(page, page * nr, scale=page)
    cont = K.ref_container(chk, data, page, wm)
    hs = K.hostile_containers(cont, page, K.chunk_pages(page, nr, 1, 1), seed=page)
    variants = [("single", "pinned", 0), ("single", "pageable", 1), ([0, 0, 0], "pageable", 3), (None, "pinned", 2),
                ([0] * 5, "no_bounce", 1)]
    with knobs(cs, chunk_mb=1, no_bounce=0):
        for k, h in enumerate(hs):
            cap = K.capacity_of(h, nr, page) if h.cls != "nr_max" else nr * page
            want = K.read_container(h.cont, page, cap)
            for devices, mem, off in (variants if k % 3 == 0 else variants[k % 5:k % 5 + 2]):
                cs.set_tuning("no_bounce", int(mem == "no_bounce"))
                got = bc_read(cs, h.cont, page, devices, "pinned" if mem == "pinned" else "pageable", off, cap)
                check_read(got, want, page, (h.name, devices, mem), untouched_after_prefix=True)


@pytest.mark.parametrize("page", [4095, 1000, 4096])
def test_container_reader_under_every_decoder_choice(cs, chk, page):
    """The reader's page slots are page_size apart, so for most page sizes they are not 16-byte aligned, which the
    lane-per-block decoder needs: forcing it (decompress_stage_input 4) must not fail the call.  Every other
    decoder choice and lane group gives the same result too."""
    nr = 800
    data = K.mixed_bytes(page + 1, page * nr - 7, scale=page)
    ref = K.ref_container(chk, data, page, 13)
    hs = [h for h in K.hostile_containers(ref, page, K.chunk_pages(page, nr), seed=3)
          if h.cls in ("two_chunks", "entry_page+1", "entry_0")][:4]
    for lanes in (32, 16, 8):
        for stage in (4, 3, 1, 2, 0):
            with knobs(cs, decompress_lanes=lanes, decompress_stage_input=stage):
                for cont in [ref] + [h.cont for h in hs]:
                    want = K.read_container(cont, page, nr * page)
                    check_read(bc_read(cs, cont, page, "single", "pinned", 0), want, page, (page, lanes, stage))


# ------------------------------------------------------------------------------------------ csnappy_batch_compress
def batch_compress(cs, bufs, wm, *, form="offsets", out_stride=None, ws_delta=0, expect_rc=0):
    """csnappy_batch_compress through ctypes, output slots pre-filled.  form: "offsets" (h_in_off, h_in_len),
    "strided" (h_in_off NULL), "uniform" (h_in_len NULL), "both" (both NULL).  -> (out numpy, out_len, stride)"""
    L = cs.api.lib()
    n = len(bufs)
    lens = np.array([len(b) for b in bufs], dtype=np.uint32)
    longest = int(lens.max()) if n else 0
    if form in ("uniform", "both"):
        assert len(set(lens.tolist())) == 1
    stride_in = longest + 7 | 1  # odd
    if form in ("strided", "both"):
        offs = np.arange(n, dtype=np.uint64) * stride_in
    else:
        offs = np.zeros(n, dtype=np.uint64)
        pos = 3
        for i, b in enumerate(bufs):
            offs[i] = pos
            pos += len(b) + 3
    total = int(offs[-1]) + longest + 64 if n else 64
    host = np.zeros(total, dtype=np.uint8)
    for o, b in zip(offs, bufs):
        host[int(o):int(o) + len(b)] = np.frombuffer(b, dtype=np.uint8)
    d_in = torch.from_numpy(host).cuda()
    bound = 5 + longest + longest // 6 + 32 * max(1, -(-longest // 32768))
    stride = bound if out_stride is None else out_stride
    out = torch.full((n * stride + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    out_len = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda")
    p_len = None if form in ("uniform", "both") else lens.ctypes.data
    p_off = None if form in ("strided", "both") else offs.ctypes.data
    uni = int(lens[0]) if form in ("uniform", "both") else 0
    ws_bytes = L.csnappy_batch_compress_workspace(p_len, uni, n)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device="cuda")
    rc = L.csnappy_batch_compress(d_in.data_ptr(), p_off, stride_in if p_off is None else 0, p_len, uni, n,
                                  out.data_ptr(), stride, out_len.data_ptr(), wm, ws.data_ptr(), ws_bytes + ws_delta,
                                  torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == expect_rc, cs.api.last_error()
    return out.cpu().numpy(), out_len.cpu().numpy().astype(np.int64), stride


def check_framed(chk, bufs, wm, out, out_len, stride, exp=None):
    n = len(bufs)
    assert (out[n * stride:] == PAT).all(), "wrote past the last slot"
    bad = []
    for i, b in enumerate(bufs):
        e = exp[i] if exp is not None else K.frame(chk, b, wm)
        slot = out[i * stride:(i + 1) * stride]
        if out_len[i] != len(e) or slot[: len(e)].tobytes() != e:
            bad.append((i, len(b), int(out_len[i]), len(e)))
        elif not (slot[len(e):] == PAT).all():
            bad.append((i, len(b), "wrote past out_len"))
        if len(bad) >= 8:
            break
    assert not bad, bad


HEADER_EDGES = [0, 1, 127, 128, 16383, 16384, 32767, 32768, 32769, (1 << 21) - 1, 1 << 21, (1 << 21) + 1]


def test_batch_compress_header_edges(cs, chk):
    src = K.mixed_bytes(21, (1 << 21) + 1 + 4099, scale=20000)
    bufs = [src[k % 4099:k % 4099 + n] for k, n in enumerate(HEADER_EDGES)]
    for wm in (9, 13, 16):
        check_framed(chk, bufs, wm, *batch_compress(cs, bufs, wm))
    # the strided and uniform forms
    small = [src[7 * k:7 * k + n] for k, n in enumerate([0, 1, 127, 128, 16384, 32769, 70000])]
    check_framed(chk, small, 13, *batch_compress(cs, small, 13, form="strided"))
    same = [src[k * 1001:k * 1001 + 40961] for k in range(5)]
    for form in ("uniform", "both", "offsets"):
        check_framed(chk, same, 15, *batch_compress(cs, same, 15, form=form))


def test_batch_compress_4_and_5_byte_headers(cs, chk):
    """2^28 - 1 and 2^28 bytes of low-entropy data in one call (0.5 GiB): the 4- and 5-byte varint headers."""
    rng = np.random.default_rng(28)
    period = np.concatenate([rng.integers(97, 101, 40961, dtype=np.uint8), np.zeros(3001, np.uint8)])
    x = np.tile(period, (1 << 28) // len(period) + 1)[: 1 << 28].tobytes()
    bufs = [x[: (1 << 28) - 1], x]
    out, out_len, stride = batch_compress(cs, bufs, 16)
    exp = [chk.compress(b, 16) for b in bufs]
    assert exp[0][:4] == bytes([0xFF, 0xFF, 0xFF, 0x7F]) and exp[1][:5] == bytes([0x80, 0x80, 0x80, 0x80, 0x01])
    check_framed(chk, bufs, 16, out, out_len, stride, exp=exp)


def test_batch_compress_many_empty_and_many_fragments(cs, chk):
    rng = np.random.default_rng(5)
    src = K.mixed_bytes(5, 300000, scale=8000)
    # thousands of empty buffers next to a few long ones: the header-only units outnumber the fragments
    lens = [0] * 5000
    for i in rng.choice(5000, 12, replace=False):
        lens[int(i)] = int(rng.integers(1, 100000))
    bufs = [src[i % 1000:i % 1000 + n] for i, n in enumerate(lens)]
    check_framed(chk, bufs, 13, *batch_compress(cs, bufs, 13))
    # more than 4096 fragments: several per scan thread
    lens = [int(rng.integers(1, 3000)) for _ in range(4500)] + [70000, 32769, 65536]
    bufs = [src[i % 5000:i % 5000 + n] for i, n in enumerate(lens)]
    assert sum(-(-n // 32768) for n in lens) > 4096
    check_framed(chk, bufs, 11, *batch_compress(cs, bufs, 11))


def test_batch_compress_refuses_short_stride_and_workspace(cs):
    bufs = [bytes(70000), b"abc"]
    bound = 5 + 70000 + 70000 // 6 + 32 * 3
    out, _, _ = batch_compress(cs, bufs, 13, out_stride=bound - 1, expect_rc=cs.api.CSNAPPY_E_BAD_ARG)
    assert (out == PAT).all()
    out, _, _ = batch_compress(cs, bufs, 13, ws_delta=-1, expect_rc=cs.api.CSNAPPY_E_BAD_ARG)
    assert (out == PAT).all()


# ------------------------------------------------------------------------------------------------ csnappy_batch_pack
def pack(cs, n, stride, base, lens, packed=True):
    L = cs.api.lib()
    gen = torch.Generator(device="cuda")
    gen.manual_seed(n * 7 + stride + base)
    slots = torch.randint(0, 256, (n * stride + base + 16,), dtype=torch.uint8, device="cuda", generator=gen)
    d_len = torch.from_numpy(lens.astype(np.int32)).cuda()
    total = int(lens.astype(np.int64).sum())
    pb = (base + 1) % 4
    out = torch.full((pb + total + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    off = torch.full((n + 1 + 8,), -0x5A5A5A5A5A5A5A5B, dtype=torch.int64, device="cuda")
    rc = L.csnappy_batch_pack(slots.data_ptr() + base if n else None, stride, d_len.data_ptr() if n else None, n,
                              (out.data_ptr() + pb) if packed else None, off.data_ptr(),
                              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0, cs.api.last_error()
    o = off.cpu().numpy()
    want = np.concatenate([[0], np.cumsum(lens.astype(np.int64))])
    assert (o[: n + 1] == want).all(), (n, stride, base)
    assert (o[n + 1:] == -0x5A5A5A5A5A5A5A5B).all(), "wrote behind off[n]"
    p = out.cpu().numpy()
    if not packed:
        assert (p == PAT).all()
        return
    assert (p[:pb] == PAT).all() and (p[pb + total:] == PAT).all(), "wrote outside the packed payload"
    s = slots.cpu().numpy()[base: base + n * stride].reshape(n, stride) if n else np.zeros((0, stride), np.uint8)
    mask = np.arange(stride)[None, :] < lens[:, None]
    assert (p[pb:pb + total] == s[mask]).all(), (n, stride, base)


@pytest.mark.parametrize("n", [0, 1, 1023, 1024, 1025, 4097])
def test_batch_pack(cs, n):
    rng = np.random.default_rng(n)
    for stride in (4813, 4816, 4817):
        lens = rng.integers(0, stride + 1, n).astype(np.int64)
        lens[: min(n, 4)] = [0, stride, 1, 3][: min(n, 4)]
        for base in range(4):
            pack(cs, n, stride, base, lens)
        pack(cs, n, stride, 1, lens, packed=False)


def test_batch_pack_200001_blocks(cs):
    n, stride = 200001, 4817
    lens = np.random.default_rng(2).integers(0, stride + 1, n).astype(np.int64)
    lens[::1000] = 0
    lens[1::1000] = stride
    pack(cs, n, stride, 3, lens)
    pack(cs, n, stride, 0, lens, packed=False)


# ------------------------------------------------------------------------------------- drop-in csnappy_compress chunks
def test_dropin_compress_chunk_edges(cs, chk):
    """Fragments go through the pipeline in chunks of 256: the last chunk holds one fragment, a 1-byte one with +1
    (the short-chunk table rule at its smallest)."""
    src = K.mixed_bytes(256, 257 * 32768, scale=32768)
    for n in (256 * 32768 - 1, 256 * 32768, 256 * 32768 + 1, 257 * 32768):
        for wm in (12, 16):
            assert cs.csnappy_compress(src[:n], wm) == chk.compress(src[:n], wm), (n, wm)


# -------------------------------------------------------------------------------------------- strided host batches
def _host_arrays(mem, shape_bytes, fill=PAT):
    t = torch.full((shape_bytes,), fill, dtype=torch.uint8)
    if mem == "pinned":
        t = t.pin_memory()
    return t, t.numpy()


def _host_words(mem, n, dtype):
    t = torch.full((n,), -7, dtype=dtype)
    if mem == "pinned":
        t = t.pin_memory()
    return t, t.numpy()


def _want_decode(port, s, cap, flags, cs):
    if flags & cs.api.BATCH_RAW_IF_FULL and len(s) == cap:
        return 0, s
    if flags & cs.api.BATCH_WITH_HEADER:
        h, olen = port.get_uncompressed_length(s)
        if h < 0:
            return h, None
        if olen > cap:
            return cs.api.CSNAPPY_E_OUTPUT_INSUF, None
        return port.decompress_noheader(s[h:], olen)
    return port.decompress_noheader(s, cap)


@pytest.mark.parametrize("mem", ["pinned", "pageable", "no_bounce"])
def test_host_batch_calls_keep_slot_tails(cs, chk, mem):
    """chunk_mb 1: 1024-block chunks, 4097 blocks, so the last chunk holds one.  Odd strides; every slot ends in a
    guard band behind the bytes the call may write (compress: csnappy_max_compressed_length of the block length;
    decompress: the capacity), and that band, and what follows the last slot, must stay as it was."""
    port = oracle.port()
    n, L, wm = 4097, 4093, 13
    src = K.mixed_bytes(4097, n * 4096, scale=4096)
    pages = [src[i * 4096:i * 4096 + L] for i in range(n)]
    km = "pageable" if mem == "no_bounce" else mem
    with knobs(cs, chunk_mb=1, no_bounce=int(mem == "no_bounce")):
        # compress: in_stride 4099, out_stride = bound + 256 (odd)
        in_stride, bound = 4099, K.max_clen(L)
        out_stride = bound + 256
        t_in, a_in = _host_arrays(km, n * in_stride, fill=0)
        a_in.reshape(n, in_stride)[:, :L] = np.frombuffer(b"".join(pages), dtype=np.uint8).reshape(n, L)
        t_out, a_out = _host_arrays(km, n * out_stride + GUARD)
        t_len, a_len = _host_words(km, n, torch.int32)
        cs.batch_compress_fragments_host(a_in, L, n, wm, a_out, a_len, in_stride=in_stride, out_stride=out_stride)
        o = a_out[: n * out_stride].reshape(n, out_stride)
        assert (a_out[n * out_stride:] == PAT).all(), "compress wrote past the last slot"
        bad = [i for i in range(n) if not (o[i, bound:] == PAT).all()]
        assert not bad, ("compress wrote past csnappy_max_compressed_length in slots", bad[:10], len(bad))
        comp = []
        for i in range(n):
            e = chk.compress_fragment(pages[i], wm)
            assert a_len[i] == len(e) and o[i, : len(e)].tobytes() == e, i
            comp.append(e)
        # decompress: in_stride 4813 (odd), cap 4096, out_stride = cap + 256 + 1; ragged lengths; failures in later
        # chunks; plain, WITH_HEADER and RAW_IF_FULL
        rng = np.random.default_rng(7)
        cap, in_stride = 4096, 4813
        out_stride = cap + 257
        for flags in (0, cs.api.BATCH_WITH_HEADER, cs.api.BATCH_RAW_IF_FULL):
            streams = []
            for i in range(n):
                body = comp[i]
                if i >= 2048 and i % 97 == 5:
                    body = bytes([0xFE, 0xFF, 0xFF]) + body[3:]  # a copy of offset 65535 before anything was produced
                s = body if flags != cs.api.BATCH_WITH_HEADER else K.varint32(L) + body
                if i >= 2048 and i % 89 == 7:
                    s = s[: len(s) // 2]
                elif flags == cs.api.BATCH_WITH_HEADER and i % 101 == 9:
                    s = K.varint32(cap + 1 + i) + comp[i]  # -2
                elif flags == cs.api.BATCH_WITH_HEADER and i % 103 == 11:
                    s = bytes([0x80] * 5)  # -1
                elif flags == cs.api.BATCH_RAW_IF_FULL and i % 7 == 3:
                    s = rng.integers(0, 256, cap, dtype=np.uint8).tobytes()  # stored: copied
                streams.append(s)
            t_in, a_in = _host_arrays(km, n * in_stride, fill=0)
            h = a_in.reshape(n, in_stride)
            for i, s in enumerate(streams):
                h[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
            t_ilen, a_ilen = _host_words(km, n, torch.int32)
            a_ilen[:] = [len(s) for s in streams]
            t_out, a_out = _host_arrays(km, n * out_stride + GUARD)
            t_olen, a_olen = _host_words(km, n, torch.int32)
            t_st, a_st = _host_words(km, n, torch.int32)
            cs.batch_decompress_host(a_in, in_stride, a_ilen, n, a_out, out_stride, cap, a_olen, a_st, flags)
            o = a_out[: n * out_stride].reshape(n, out_stride)
            assert (a_out[n * out_stride:] == PAT).all(), ("decompress wrote past the last slot", flags)
            bad = [i for i in range(n) if not (o[i, cap:] == PAT).all()]
            assert not bad, ("decompress wrote at or past cap in slots", flags, bad[:10], len(bad))
            n_err = 0
            for i, s in enumerate(streams):
                rc, e = _want_decode(port, s, cap, flags, cs)
                assert a_st[i] == rc, (flags, i)
                if rc == 0:
                    assert a_olen[i] == len(e) and o[i, : len(e)].tobytes() == e, (flags, i)
                else:
                    n_err += 1
                    assert a_olen[i] == 0, (flags, i)
            assert n_err >= 20 and all(_want_decode(port, streams[i], cap, flags, cs)[0] == 0 for i in range(2048)
                                       if not (flags == cs.api.BATCH_WITH_HEADER and (i % 101 == 9 or i % 103 == 11)))
