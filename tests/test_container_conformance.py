"""The restated page container, reader and csnappy_compress framing (tests/containers.py) against the oracle port,
and the coverage of the generated inputs.

The GPU framing tests compare the container calls, csnappy_batch_compress and the drop-in framing with these
restatements; that is only worth something if the restatements agree with the reference and the inputs reach the
edges: pages whose compressed size is page + 1, page and page - 1 at every page size, stored short last pages,
last chunks of one page, and every class of broken index."""
import os
import struct
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import containers as K  # noqa: E402
import oracle  # noqa: E402

# page size -> table size of the GPU file (any of 9..16 fits every page size)
PAGES = {1: 9, 3: 10, 17: 11, 64: 12, 1000: 13, 4095: 14, 4096: 13, 4097: 15, 16384: 16, 20000: 14, 32767: 15,
         32768: 16}


@pytest.fixture(scope="module")
def port():
    return oracle.port()


@pytest.mark.parametrize("page", [p for p in PAGES if p >= 64])
def test_equality_pages_found_at_every_page_size(port, page):
    wm = PAGES[page]
    eq = K.equality_pages(page, wm)
    assert sorted(eq) == ([-1, 0] if page == 64 else [-1, 0, 1]), (page, sorted(eq))
    for d, p in eq.items():
        assert len(p) == page and len(port.compress_fragment(p, wm)) == page + d


@pytest.mark.parametrize("page", list(PAGES))
def test_writer_and_reader_round_trip_every_generated_input(port, page):
    wm = PAGES[page]
    tail = 1 + page % 31 if page > 31 else 0
    data, cls = K.container_input(page, wm, seed=5, tail=tail)
    if page >= 64:
        assert {"eq+0", "eq-1"} | ({"eq+1"} if page > 64 else set()) <= set(cls)
    inputs = [data, bytes(page * 300 + 7), np.random.default_rng(page).integers(0, 256, page * 40, dtype=np.uint8).tobytes(),
              K.mixed_bytes(page, page * 300 + page // 2, scale=max(page, 64))]
    for n in K.edge_lengths(page, ks=(1,)):
        inputs.append(K.mixed_bytes(n, n, scale=max(page, 64)))
    for x in inputs:
        cont = K.ref_container(port, x, page, wm)
        nr = (len(x) + page - 1) // page
        idx = np.frombuffer(cont, dtype="<u4", count=nr, offset=4)
        assert (idx <= page).all()
        r = K.read_container(cont, page, nr * page)
        full = [i for i in range(nr) if i < nr - 1 or len(x) % page == 0]
        if len(x) % page == 0 or int(idx[-1]) < len(x) % page:
            # every page round-trips when the last page is whole or compressed
            assert r.key() == (0, len(x), None), (page, len(x))
            assert b"".join(r.pages[i] for i in range(nr)) == x
        else:
            # a stored short last page is decoded as Snappy: the reference's wart
            last = x[(nr - 1) * page:]
            rc, out = port.decompress_noheader(last, page)
            assert r.rc == rc and r.failed_page == (None if rc == 0 else nr - 1)
            assert r.out_length == page * (nr - 1) + (len(out) if rc == 0 else 0)
        assert all(r.pages[i] == x[i * page:(i + 1) * page] for i in full)
    # the equality pages: page - 1 is kept compressed, page and page + 1 are stored
    if page >= 64:
        cont = K.ref_container(port, data, page, wm)
        idx = np.frombuffer(cont, dtype="<u4", offset=4, count=(len(data) + page - 1) // page)
        assert [int(idx[cls[k][0]]) for k in ("eq+1", "eq+0", "eq-1") if k in cls] == [page, page, page - 1][page == 64:]


def test_stored_short_last_page_reads_as_the_oracle_decodes_it(port):
    """Stored tails of 1..31 bytes: the reader's result for the last page is the oracle's raw decode of them.
    Random tails fail; a tail that happens to be a Snappy literal decodes to one byte less than was written."""
    page = 4096
    rcs = set()
    for n, snappy in [(n, s) for n in range(1, 32) for s in (False, True)]:
        tail = K.short_tail(9, n, snappy)
        data = bytes(2 * page) + tail
        cont = K.ref_container(port, data, page, 13)
        assert struct.unpack_from("<I", cont, 12)[0] == n  # stored: entry = its length, below the page size
        r = K.read_container(cont, page, 3 * page)
        rc, out = port.decompress_noheader(tail, page)
        rcs.add(rc)
        assert (r.rc, r.failed_page) == ((rc, None) if rc == 0 else (rc, 2))
        if rc == 0:
            assert r.pages[2] == out and r.out_length == 2 * page + len(out)
            assert out == tail[1:] or n == 1
    assert {0, K.E_DATA_MALFORMED} <= rcs, rcs


@pytest.mark.parametrize("wm", [9, 13, 16])
def test_framing_restatement_equals_port(port, wm):
    rng = np.random.default_rng(wm)
    src = K.mixed_bytes(wm, 3 * 32768 + 5000, scale=20000)
    for n in (0, 1, 127, 128, 129, 255, 256, 257, 16383, 16384, 32767, 32768, 32769, 65535, 65536, 65537,
              2 * 32768 + 4097, 3 * 32768 + 1):
        assert K.frame(port, src[:n], wm) == port.compress(src[:n], wm), (n, wm)
    for n in (1 << 21) - 1, 1 << 21, (1 << 21) + 1:
        x = np.tile(rng.integers(97, 101, 4099, dtype=np.uint8), n // 4099 + 1)[:n].tobytes()
        assert K.frame(port, x, wm) == port.compress(x, wm), n
    assert [K.header_length(n) for n in (0, 127, 128, 16383, 16384, (1 << 21) - 1, 1 << 21, (1 << 28) - 1, 1 << 28)] == \
        [1, 1, 2, 2, 3, 3, 4, 4, 5]
    assert all(K.chunk_wm(n, w) == port.chunk_wm(n, w) for w in range(9, 17)
               for n in (1, 255, 256, 257, 4096, 4097, 16384, 32767, 32768))


def test_edge_lengths_put_one_page_in_the_last_chunk():
    for page in PAGES:
        for workers in (1, 3):
            for mb in (0, 1):
                lasts = set()
                for n in K.edge_lengths(page):
                    nr = (n + page - 1) // page
                    chunk = K.chunk_pages(page, nr, workers, mb)
                    assert chunk == min(K.CHUNK_MIN, nr), (page, n, workers, mb, chunk)
                    lasts.add(nr - (nr - 1) // chunk * chunk)
                assert {1, K.CHUNK_MIN} <= lasts, (page, lasts)


@pytest.mark.parametrize("page", [4096, 1000])
def test_hostile_containers_cover_every_class(port, page):
    wm = PAGES[page]
    data = K.mixed_bytes(page, page * 1100, scale=page)
    cont = K.ref_container(port, data, page, wm)
    chunk = K.chunk_pages(page, 1100, 1, 1)
    hs = K.hostile_containers(cont, page, chunk, seed=page)
    assert {h.cls for h in hs} == K.HOSTILE_CLASSES
    nr = 1100
    codes = {}
    for h in hs:
        r = K.read_container(h.cont, page, K.capacity_of(h, nr, page))
        codes[h.cls] = r
    assert codes["nr_0"].key() == (0, 0, None)
    assert codes["nr_max"].key() == (K.E_DATA_MALFORMED, 0, None)
    assert codes["capacity"].key() == (K.E_OUTPUT_INSUF, 0, None)
    # the smallest failing page wins, whichever kind of failure it is
    two = next(h for h in hs if h.cls == "two_chunks")
    a, b = (int(x) for x in two.name.split("pages ")[1].split(" and "))
    assert codes["two_chunks"].failed_page == a and codes["one_failure"].failed_page == b
    assert a // chunk != b // chunk
    assert codes["index_before_decode"].key()[::2] == (K.E_DATA_MALFORMED, a)
    assert codes["index_before_decode"].prefix == a
    assert codes["index_after_decode"].failed_page == a and codes["index_after_decode"].prefix == b
    # pages behind a failure are decoded and counted
    assert codes["one_failure"].out_length == page * (nr - 1)
    for h in hs:
        if h.cls.startswith("entry_max_clen+1"):
            assert codes[h.cls].rc == K.E_DATA_MALFORMED
