"""The page container on device buffers (csnappy_bc_compress, csnappy_bc_index, csnappy_bc_decompress_pages,
csnappy_bc_decompress) against the restatements of tests/containers.py and against the host container calls.

  writer       page sizes 1 ... 32768, edge lengths and empty input, wm 9-16, input and container at byte offsets 0, 1, 3
               and 13; a guard pattern around the container slot.
  whole reader valid containers and every class of containers.hostile_containers, at odd container offsets; pages past
               the decodable prefix stay unwritten; a container of 160 Ki 4 KiB pages (above the lane decoder's
               threshold) under every decoder routing; two reads on two streams at once.
  index        offsets against the restated index scan, a short index, an index too small for the count, and a
               5 Mi-entry index (more tiles than the tile scan's threads).
  page reads   permutations, duplicates, no requests, page numbers >= nr, pages behind a malformed entry, pages that
               fail to decode, stored full and short last pages, out_stride equal to and above an odd page size; the
               launch count of 1 and of 100 000 requests.
Each request's expected (status, bytes) comes from the restated index scan and an oracle decode of its payload.
"""
import ctypes as C
import os
import struct
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
NO_PAGE = 2**64 - 1
OFFSETS = (0, 1, 3, 13)


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.fixture(scope="module")
def chk():
    return oracle.best()


def stream():
    return torch.cuda.current_stream().cuda_stream


def dev_at(data: bytes, off: int):
    """data at byte `off` of a pattern-filled CUDA allocation with a guard band behind it -> (tensor, pointer)."""
    t = torch.full((off + len(data) + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    if data:
        t[off:off + len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    return t, t.data_ptr() + off


# ------------------------------------------------------------------------------------------------- restatements
def restated_index(cont: bytes, page: int):
    """-> (nr, [payload offset or NO_PAGE per page]) by the host reader's index scan."""
    nr = struct.unpack_from("<I", cont, 0)[0]
    idx = np.frombuffer(cont, dtype="<u4", count=nr, offset=4).astype(np.int64)
    out = [NO_PAGE] * nr
    pos = 4 + 4 * nr
    for i in range(nr):
        cl = int(idx[i])
        if cl > K.max_clen(page) or pos + cl > len(cont):
            break
        out[i] = pos
        pos += cl
    return nr, out


def restated_request(cont: bytes, page: int, offs, p: int, nr: int):
    """Expected (status, bytes) of one page request."""
    if p >= nr:
        return K.E_BAD_ARG, None
    if offs[p] == NO_PAGE:
        return K.E_DATA_MALFORMED, None
    cl = struct.unpack_from("<I", cont, 4 + 4 * p)[0]
    payload = cont[offs[p]:offs[p] + cl]
    if cl == page:
        return 0, payload
    rc, out = oracle.port().decompress_noheader(payload, page)
    return rc, (out if rc == 0 else None)


# ------------------------------------------------------------------------------------------------------ callers
def dev_write(cs, data: bytes, page: int, wm: int, in_off: int, out_off: int):
    """csnappy_bc_compress -> (container bytes, whole container allocation as numpy, container length)"""
    L = cs.api.lib()
    cap = L.csnappy_bc_max_container_length(len(data), page)
    d_in, p_in = dev_at(data, in_off)
    cont = torch.full((out_off + cap + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    length = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    ws_n = L.csnappy_bc_compress_workspace(len(data), page)
    ws = torch.empty(max(ws_n, 1), dtype=torch.uint8, device="cuda")
    rc = L.csnappy_bc_compress(p_in, len(data), page, cont.data_ptr() + out_off, cap, length.data_ptr(), wm,
                               ws.data_ptr(), ws_n, stream())
    assert rc == 0, cs.api.last_error()
    torch.cuda.synchronize()
    a = cont.cpu().numpy()
    n = int(length.item())
    return a[out_off:out_off + n].tobytes(), a, n


def dev_read(cs, cont: bytes, page: int, cap: int, off: int = 0, s=None, keep=None):
    """csnappy_bc_decompress -> (rc, out_length, failed_page or None, output [0, cap) as numpy).  Checks that nothing is
    written behind cap and that failed_page is written only on a page failure."""
    L = cs.api.lib()
    d, p = dev_at(cont, off)
    out = torch.full((cap + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    olen = torch.full((1,), -7, dtype=torch.int64, device="cuda")
    words = torch.full((2,), -1, dtype=torch.int32, device="cuda")
    ws_n = L.csnappy_bc_decompress_workspace(len(cont), page, cap)
    ws = torch.empty(max(ws_n, 1), dtype=torch.uint8, device="cuda")
    rc = L.csnappy_bc_decompress(p, len(cont), page, out.data_ptr(), cap, olen.data_ptr(), words.data_ptr(),
                                 words.data_ptr() + 4, ws.data_ptr(), ws_n, s if s is not None else stream())
    assert rc == 0, cs.api.last_error()
    if keep is not None:  # concurrent use: the caller synchronises
        keep.append((d, out, olen, words, ws))
        return out, olen, words
    torch.cuda.synchronize()
    return unpack_read(out, olen, words, cap)


def unpack_read(out, olen, words, cap):
    a = out.cpu().numpy()
    assert (a[cap:] == PAT).all(), "whole-container reader wrote past out_capacity"
    st, bad = (int(x) for x in words.cpu().tolist())
    if st == 0:
        assert bad == -1, "failed_page written on success"
    return st, int(olen.item()), (bad & 0xFFFFFFFF if bad != -1 else None), a[:cap]


def host_read(cs, cont: bytes, page: int, cap: int):
    L = cs.api.lib()
    src = np.frombuffer(cont, dtype=np.uint8) if cont else np.zeros(1, np.uint8)
    out = np.zeros(max(cap, 1), dtype=np.uint8)
    olen, bad = C.c_uint64(0), C.c_uint32(0xFFFFFFFF)
    rc = L.csnappy_bc_decompress_host(src.ctypes.data, len(cont), page, out.ctypes.data, cap, C.byref(olen),
                                      C.byref(bad))
    return rc, olen.value, (bad.value if rc != 0 and bad.value != 0xFFFFFFFF else None)


def dev_index(cs, cont: bytes, page: int, off: int = 0, entries=None):
    """csnappy_bc_index -> (rc, nr, index list or None)"""
    L = cs.api.lib()
    d, p = dev_at(cont, off)
    nr = C.c_uint32(0xDEADBEEF)
    n = entries if entries is not None else max((len(cont) - 4) // 4, 0)
    idx = torch.full((max(n, 1) + 4,), -3, dtype=torch.int64, device="cuda")
    rc = L.csnappy_bc_index(p, len(cont), page, idx.data_ptr(), n, C.byref(nr), stream())
    torch.cuda.synchronize()
    if rc != 0:
        return rc, nr.value, None
    got = [int(x) & (2**64 - 1) for x in idx[: nr.value].cpu().tolist()]
    assert (idx[nr.value:] == -3).all(), "index written past nr_pages"
    return rc, nr.value, got


def dev_pages(cs, cont: bytes, page: int, pages, out_stride: int, off: int = 0):
    """index + csnappy_bc_decompress_pages -> (out numpy, out_len, status), guard bytes between slots checked"""
    L = cs.api.lib()
    d, p = dev_at(cont, off)
    nr = C.c_uint32(0)
    n_idx = max((len(cont) - 4) // 4, 1)
    idx = torch.empty(n_idx, dtype=torch.int64, device="cuda")
    assert L.csnappy_bc_index(p, len(cont), page, idx.data_ptr(), n_idx, C.byref(nr), stream()) == 0, cs.api.last_error()
    k = len(pages)
    pg = torch.tensor(np.asarray(pages, dtype=np.uint32).view(np.int32), dtype=torch.int32).cuda() if k else \
        torch.empty(1, dtype=torch.int32, device="cuda")
    out = torch.full((max(k * out_stride, 1) + GUARD,), PAT, dtype=torch.uint8, device="cuda")
    olen = torch.full((max(k, 1),), -9, dtype=torch.int32, device="cuda")
    st = torch.full((max(k, 1),), -9, dtype=torch.int32, device="cuda")
    ws_n = L.csnappy_bc_decompress_pages_workspace(k)
    ws = torch.empty(ws_n, dtype=torch.uint8, device="cuda")
    rc = L.csnappy_bc_decompress_pages(p, len(cont), page, idx.data_ptr(), nr.value, pg.data_ptr(), k, out.data_ptr(),
                                       out_stride, olen.data_ptr(), st.data_ptr(), ws.data_ptr(), ws_n, stream())
    assert rc == 0, cs.api.last_error()
    torch.cuda.synchronize()
    a = out.cpu().numpy()
    assert (a[k * out_stride:] == PAT).all(), "page reads wrote past the last slot"
    for j in range(k):
        assert (a[j * out_stride + page:(j + 1) * out_stride] == PAT).all(), ("wrote between slots", j)
    return a, olen.cpu().numpy()[:k], st.cpu().numpy()[:k], nr.value


def check_pages(cont, page, pages, got, out_stride, what):
    a, olen, st, nr = got
    n2, offs = restated_index(cont, page)
    assert nr == n2
    for j, p in enumerate(pages):
        rc, b = restated_request(cont, page, offs, int(p), nr)
        assert int(st[j]) == rc, (what, j, int(p), int(st[j]), rc)
        if rc == 0:
            assert int(olen[j]) == len(b), (what, j, int(p))
            assert a[j * out_stride:j * out_stride + len(b)].tobytes() == b, (what, "bytes", j, int(p))
        else:
            assert int(olen[j]) == 0, (what, j)


def check_whole(cs, cont, page, cap, got, what):
    rc, olen, bad, out = got
    want = K.read_container(cont, page, cap)
    assert (rc, olen, bad) == want.key(), (what, (rc, olen, bad), want.key())
    assert host_read(cs, cont, page, cap) == want.key(), (what, "host call")
    for i, b in want.pages.items():
        assert out[i * page:i * page + len(b)].tobytes() == b, (what, "page", i)
    assert (out[want.prefix * page:] == PAT).all(), (what, "wrote a page past the decodable prefix")


# ---------------------------------------------------------------------------------------------------- writer
@pytest.mark.parametrize("page", [1, 13, 64, 4095, 4096, 4097, 32768])
def test_writer_bytes(cs, chk, page):
    tail = 1 + page % 31 if page > 31 else 0
    base, _ = K.container_input(page, 13, seed=5, tail=tail)
    inputs = [(base, wm) for wm in range(9, 17)]
    inputs += [(K.mixed_bytes(50 + j, n, scale=max(page, 64)), 9 + (j * 3) % 8)
               for j, n in enumerate(K.edge_lengths(page, ks=(1,)))]
    inputs.append((b"", 13))
    if page > 31:
        inputs.append((base[:len(base) - tail] + K.short_tail(9, tail, snappy=True), 11))
    for k, (x, wm) in enumerate(inputs):
        ref = K.ref_container(chk, x, page, wm)
        io, oo = OFFSETS[k % 4], OFFSETS[(k + 1 + k // 4) % 4]
        got, alloc, n = dev_write(cs, x, page, wm, io, oo)
        what = (page, len(x), wm, io, oo)
        assert n == len(ref), what
        assert got == ref, what
        assert (alloc[:oo] == PAT).all() and (alloc[oo + n:] == PAT).all(), (what, "wrote outside the container")
        if k % 5 == 0:
            cont = np.zeros(cs.api.bc_max_container_length(len(x), page), dtype=np.uint8)
            src = np.frombuffer(x, dtype=np.uint8) if x else np.zeros(1, np.uint8)
            clen = cs.api.bc_compress_host(src, len(x), cont, wm, page)
            assert cont[:clen].tobytes() == got, (what, "host call")


def test_writer_python_api(cs, chk):
    data = K.mixed_bytes(77, 300 * 4096 + 17)
    d = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    out, length = cs.bc_compress_device(d, wm=12)
    torch.cuda.synchronize()
    ref = K.ref_container(chk, data, 4096, 12)
    assert int(length.item()) == len(ref) and out[:len(ref)].cpu().numpy().tobytes() == ref
    rc, idx, nr = cs.bc_index_device(out, len(ref))
    assert rc == 0 and nr == 301 and [int(x) & (2**64 - 1) for x in idx.cpu().tolist()] == restated_index(ref, 4096)[1]
    back, res = cs.bc_decompress_device(out, len(ref))
    torch.cuda.synchronize()
    assert res.cpu().tolist() == [len(data), 0, -1]
    assert back[:len(data)].cpu().numpy().tobytes() == data
    pages = torch.tensor([300, 0, 7, 7, 301], dtype=torch.int32).cuda()
    o, ol, st = cs.bc_decompress_pages_device(out, idx, nr, pages, container_length=len(ref))
    torch.cuda.synchronize()
    assert st.cpu().tolist() == [0, 0, 0, 0, K.E_BAD_ARG]
    assert ol.cpu().tolist() == [17, 4096, 4096, 4096, 0]
    o = o.cpu().numpy()
    assert o[:17].tobytes() == data[300 * 4096:] and o[2 * 4096:3 * 4096].tobytes() == data[7 * 4096:8 * 4096]


# ---------------------------------------------------------------------------------------------- whole reader
@pytest.mark.parametrize("page", [4096, 1000, 4095])
def test_whole_reader_valid_and_hostile(cs, chk, page):
    nr = 1100
    data = K.mixed_bytes(page + 3, page * nr, scale=page)
    cont = K.ref_container(chk, data, page, 13)
    hs = K.hostile_containers(cont, page, K.chunk_pages(page, nr, 1, 1), seed=page)
    seen = set()
    base, _ = K.container_input(page, 13, seed=8, tail=1 + page % 31)
    for k, c in enumerate([cont, K.ref_container(chk, base, page, 13)]):
        n = struct.unpack_from("<I", c, 0)[0]
        check_whole(cs, c, page, n * page, dev_read(cs, c, page, n * page, OFFSETS[k + 1]), ("valid", k))
    for k, h in enumerate(hs):
        seen.add(h.cls)
        cap = K.capacity_of(h, nr, page)
        got = dev_read(cs, h.cont, page, cap, OFFSETS[k % 4])
        check_whole(cs, h.cont, page, cap, got, h.name)
    assert seen == K.HOSTILE_CLASSES


def test_both_decoder_families_and_every_routing(cs):
    """160 Ki 4 KiB pages (above 148 * 1100 blocks, where the default routing takes the lane-per-block decoder) and a
    page size that is not a multiple of 16, under decompress_stage_input 0..4, against the host reader."""
    from csnappy_b200 import synth

    for page, nr in ((4096, 160 * 1024 + 100), (4095, 3000)):
        d = synth.mixed_pages(nr, page, seed=0x5EED0001 + page)
        data = d.cpu().numpy()
        cont, length = cs.bc_compress_device(d, wm=13, page_size=page)
        torch.cuda.synchronize()
        n = int(length.item())
        good = cont[:n].cpu().numpy().tobytes()
        hcont = np.zeros(cs.api.bc_max_container_length(data.size, page), dtype=np.uint8)
        assert cs.api.bc_compress_host(data, data.size, hcont, 13, page) == n and hcont[:n].tobytes() == good
        # two decode failures and a malformed entry near the end
        off = restated_index(good, page)[1]
        b = bytearray(good)
        lens = np.frombuffer(good, dtype="<u4", count=nr, offset=4)
        comp = [i for i in range(nr) if 8 < lens[i] < page]
        for i in (comp[len(comp) // 3], comp[2 * len(comp) // 3]):
            b[off[i]:off[i] + 3] = bytes([0xFE, 0xFF, 0xFF])
        b[4 + 4 * (nr - 5):8 + 4 * (nr - 5)] = struct.pack("<I", K.max_clen(page) + 1)
        bad = bytes(b)
        want_bad = host_read(cs, bad, page, nr * page)
        assert want_bad[0] != 0
        for stage in (0, 1, 2, 3, 4):
            cs.set_tuning("decompress_stage_input", stage)
            try:
                rc, olen, fp, out = dev_read(cs, good, page, nr * page)
                assert (rc, olen, fp) == (0, data.size, None), (page, stage)
                assert np.array_equal(out[:data.size], data), (page, stage)
                rc, olen, fp, out = dev_read(cs, bad, page, nr * page, off=1)
                assert (rc, olen, fp) == want_bad, (page, stage, (rc, olen, fp), want_bad)
                assert (out[(nr - 5) * page:] == PAT).all()
            finally:
                cs.set_tuning("decompress_stage_input", 0)


def test_two_streams_at_once(cs, chk):
    page, nr = 4096, 1100
    cont = K.ref_container(chk, K.mixed_bytes(11, page * nr), page, 13)
    hs = K.hostile_containers(cont, page, K.chunk_pages(page, nr, 1, 1), seed=2)
    a = next(h for h in hs if h.cls == "two_chunks").cont
    single = [dev_read(cs, c, page, nr * page) for c in (cont, a)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    keep = []
    torch.cuda.synchronize()
    r1 = dev_read(cs, cont, page, nr * page, s=s1.cuda_stream, keep=keep)
    r2 = dev_read(cs, a, page, nr * page, s=s2.cuda_stream, keep=keep)
    torch.cuda.synchronize()
    for got, want in zip((unpack_read(*r1, nr * page), unpack_read(*r2, nr * page)), single):
        assert got[:3] == want[:3] and np.array_equal(got[3], want[3])


# ------------------------------------------------------------------------------------------------------ index
def test_index_against_the_restated_scan(cs, chk):
    page, nr = 1000, 1100
    cont = K.ref_container(chk, K.mixed_bytes(21, page * nr, scale=page), page, 13)
    hs = K.hostile_containers(cont, page, K.chunk_pages(page, nr, 1, 1), seed=4)
    for k, h in enumerate([K.Hostile("valid", "valid", cont)] + hs):
        off = OFFSETS[k % 4]
        rc, n, got = dev_index(cs, h.cont, page, off)
        n2 = struct.unpack_from("<I", h.cont, 0)[0]
        if len(h.cont) < 4 + 4 * n2:
            assert (rc, n) == (K.E_DATA_MALFORMED, n2), h.name
            continue
        assert rc == 0 and n == n2, h.name
        assert got == restated_index(h.cont, page)[1], h.name
    # an index too small for the count: refused with the count set; 0 entries and no index ask for the count alone
    rc, n, _ = dev_index(cs, cont, page, 3, entries=nr - 1)
    assert (rc, n) == (K.E_BAD_ARG, nr)
    nrv = C.c_uint32(0)
    d, p = dev_at(cont, 0)
    assert cs.api.lib().csnappy_bc_index(p, len(cont), page, None, 0, C.byref(nrv), stream()) == K.E_BAD_ARG
    assert nrv.value == nr


def test_index_of_millions_of_entries(cs):
    """5 Mi entries: more tiles (4096 entries each) than the tile scan's 1024 threads; an entry above the bound and a
    payload past the end, each in a different run."""
    rng = np.random.default_rng(5)
    page, nr = 4096, 5 * 1024 * 1024 + 77
    lens = rng.integers(0, 4200, nr).astype(np.uint32)
    lens[rng.random(nr) < 0.2] = page
    head = 4 + 4 * nr
    ends = head + np.cumsum(lens.astype(np.int64))
    full = int(ends[-1])
    for case in ("valid", "big", "short"):
        ln = lens.copy()
        length = full
        if case == "big":
            ln[3_000_001] = K.max_clen(page) + 1
            length = full + K.max_clen(page)
        elif case == "short":
            length = int(ends[4_444_444]) - 1
        buf = np.concatenate((np.array([nr], dtype="<u4"), ln)).view(np.uint8)
        for off in (0, 3):
            d = torch.zeros(off + buf.size + 8, dtype=torch.uint8, device="cuda")
            d[off:off + buf.size] = torch.from_numpy(buf.copy()).cuda()
            idx = torch.empty(nr, dtype=torch.int64, device="cuda")
            nrv = C.c_uint32(0)
            assert cs.api.lib().csnappy_bc_index(d.data_ptr() + off, length, page, idx.data_ptr(), nr, C.byref(nrv),
                                                 stream()) == 0
            got = idx.cpu().numpy()
            starts = head + np.concatenate(([0], np.cumsum(ln.astype(np.int64))[:-1]))
            bad = (ln > K.max_clen(page)) | (starts + ln > length)
            first = int(np.argmax(bad)) if bad.any() else nr
            want = np.where(np.arange(nr) < first, starts, -1)
            assert np.array_equal(got, want), (case, off, first)
            assert first == {"valid": nr, "big": 3_000_001, "short": 4_444_444}[case]


# ------------------------------------------------------------------------------------------------- page reads
def test_page_reads(cs, chk):
    rng = np.random.default_rng(9)
    for page in (4096, 4095):
        tail = 1 + page % 31
        base, cls = K.container_input(page, 13, seed=12, tail=tail)
        more = K.mixed_bytes(31, page * 1200, scale=page)
        data = more + base
        cont = K.ref_container(chk, data, page, 13)
        nr = struct.unpack_from("<I", cont, 0)[0]
        snappy_tail = K.ref_container(chk, data[:len(data) - tail] + K.short_tail(4, tail, snappy=True), page, 13)
        hs = K.hostile_containers(cont, page, K.chunk_pages(page, nr, 1, 1), seed=7)
        picks = {h.cls: h.cont for h in hs if h.cls in ("index_before_decode", "two_chunks", "random_payload",
                                                          "entry_max_clen+1", "past_end_middle")}
        stored = [len(more) // page + i for i in cls["random"]]
        sets = [
            ("permutation", cont, rng.permutation(nr)),
            ("duplicates", cont, np.concatenate((rng.integers(0, nr, 500), [nr - 1] * 3 + stored * 2))),
            ("none", cont, np.zeros(0, dtype=np.int64)),
            ("beyond", cont, np.array([nr, nr + 1, 2**32 - 1, 0, nr - 1, 5 * nr])),
            ("snappy short tail", snappy_tail, np.array([nr - 1, nr - 2, nr - 1])),
        ]
        for name, c in picks.items():
            sets.append((name, c, rng.permutation(nr)[:400].tolist() + list(range(nr - 40, nr))))
        for k, (name, c, pages) in enumerate(sets):
            for stride in ((page, page + 16 + 3 * (page % 2)) if k % 2 == 0 else (page + 7,)):
                got = dev_pages(cs, c, page, list(pages), stride, OFFSETS[k % 4])
                check_pages(c, page, list(pages), got, stride, (page, name, stride))


def test_page_read_launch_count_does_not_grow(cs, chk):
    page, nr = 4096, 600
    cont = K.ref_container(chk, K.mixed_bytes(41, page * nr), page, 13)
    counts = []
    for k in (1, 100_000):
        pages = np.random.default_rng(k).integers(0, nr, k)
        before = cs.api.kernel_launches()
        got = dev_pages(cs, cont, page, list(pages), page)
        counts.append(cs.api.kernel_launches() - before)
        if k == 1:
            check_pages(cont, page, list(pages), got, page, "one request")
        else:
            assert (got[2] == 0).all()
    assert counts[0] == counts[1], counts
