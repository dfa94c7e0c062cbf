"""Plain restatements of the page container, its reader, csnappy_compress framing and the pipelines' chunking, and
seeded generators of the inputs where those go wrong.  Plain Python on top of the oracle port; no torch.

* ``ref_container``  block_compressor's writer loop (block_compressor.c:275-345): per page the fragment or, when that
  is not smaller, the page itself, behind [u32 nr][u32 clen[nr]].
* ``read_container`` the documented reader (include/csnappy_batch.h): argument checks, the index scan that ends the
  decodable prefix, a raw copy for clen == page, a raw decode for anything else, the smallest failing page wins.
  A stored SHORT last page (clen < page) is decoded as Snappy: the reference's wart, kept on both sides.
* ``frame``          csnappy_compress (csnappy_compress.c:621-656): varint32 length, then 32 KiB fragments, the short
  last one with the smaller table of ``chunk_wm``.
* ``chunk_pages``    how many pages one chunk of the container pipelines holds (csnappy_shim.c chunk_units), so that
  cases can be put at chunk edges.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field

import numpy as np

import oracle

FRAGMENT = 32768
E_OUTPUT_INSUF, E_DATA_MALFORMED, E_BAD_ARG = -2, -5, -101


def max_clen(n: int) -> int:
    return 32 + n + n // 6


def varint32(n: int) -> bytes:
    out = bytearray()
    while n >= 128:
        out.append((n & 0x7F) | 0x80)
        n >>= 7
    out.append(n)
    return bytes(out)


# ----------------------------------------------------------------------------------------------- writer and reader
def ref_container(chk, data: bytes, page: int, wm: int) -> bytes:
    """block_compressor.c:275-345 restated with `chk` as the page compressor."""
    nr = (len(data) + page - 1) // page
    idx, payload = [], []
    for i in range(nr):
        p = data[i * page:(i + 1) * page]
        c = chk.compress_fragment(p, wm)
        if len(c) >= len(p):
            c = p
        idx.append(len(c))
        payload.append(c)
    return struct.pack("<I", nr) + b"".join(struct.pack("<I", x) for x in idx) + b"".join(payload)


@dataclass
class ReadResult:
    rc: int
    out_length: int
    failed_page: int | None
    pages: dict = field(default_factory=dict)  # page index -> bytes produced, for every page that decoded
    prefix: int = 0  # pages the reader decodes (the index scan's prefix)

    def key(self):
        return self.rc, self.out_length, self.failed_page


def read_container(cont: bytes, page: int, out_capacity: int, decode=None) -> ReadResult:
    """The container reader's contract.  decode(payload, cap) -> (rc, bytes or None); default: the oracle port."""
    decode = decode or oracle.port().decompress_noheader
    if not 1 <= page <= FRAGMENT or len(cont) < 4:
        return ReadResult(E_BAD_ARG, 0, None)
    nr = struct.unpack_from("<I", cont, 0)[0]
    if len(cont) < 4 + 4 * nr:
        return ReadResult(E_DATA_MALFORMED, 0, None)
    if out_capacity < nr * page:
        return ReadResult(E_OUTPUT_INSUF, 0, None)
    idx = np.frombuffer(cont, dtype="<u4", count=nr, offset=4).astype(np.int64)
    pos = 4 + 4 * nr
    fails = []
    spans = []
    for i in range(nr):
        cl = int(idx[i])
        if cl > max_clen(page) or pos + cl > len(cont):
            fails.append((i, E_DATA_MALFORMED))
            break
        spans.append((pos, cl))
        pos += cl
    res = ReadResult(0, 0, None, prefix=len(spans))
    for i, (at, cl) in enumerate(spans):
        payload = cont[at:at + cl]
        if cl == page:
            rc, out = 0, payload
        else:
            rc, out = decode(payload, page)
        if rc == 0:
            res.pages[i] = out
            res.out_length += len(out)
        else:
            fails.append((i, rc))
    if fails:
        res.failed_page, res.rc = min(fails)
    return res


# ----------------------------------------------------------------------------------------------------- framing
def chunk_wm(n: int, wm: int) -> int:
    """The table size csnappy_compress takes for a chunk of n bytes (csnappy_compress.c:638-646)."""
    if n >= FRAGMENT:
        return wm
    ws = 9
    while ws < wm and (1 << (ws - 1)) < n:
        ws += 1
    return ws


def frame(chk, data: bytes, wm: int) -> bytes:
    parts = [varint32(len(data))]
    for at in range(0, len(data), FRAGMENT):
        c = data[at:at + FRAGMENT]
        parts.append(chk.compress_fragment(c, chunk_wm(len(c), wm)))
    return b"".join(parts)


def header_length(n: int) -> int:
    return len(varint32(n))


# -------------------------------------------------------------------------------------------- pipeline chunking
def chunk_pages(page: int, nr: int, workers: int = 1, chunk_mb: int = 0) -> int:
    """Pages per chunk of the container pipelines (csnappy_shim.c chunk_units): chunk_mb MiB (0: 32), at most a
    quarter of a worker's pages, at least 256, at most all."""
    units = ((chunk_mb or 32) << 20) // page
    per_dev = (nr + workers - 1) // workers
    units = min(units, (per_dev + 3) // 4)
    units = max(units, 256)
    return min(units, nr)


# -------------------------------------------------------------------------------------------------- generators
def mixed_bytes(seed: int, n: int, scale: int = 4096) -> bytes:
    """Segments of random bytes, 4-letter text, zeros and repeated words, of random lengths up to 3 * scale: some
    pages of a page container compress, some are stored."""
    rng = np.random.default_rng(seed)
    parts, total = [], 0
    words = [bytes(rng.integers(97, 123, int(rng.integers(3, 9)), dtype=np.uint8)) for _ in range(40)]
    while total < n:
        m = int(rng.integers(1, 3 * scale + 1))
        kind = int(rng.integers(0, 4))
        if kind == 0:
            s = rng.integers(0, 256, m, dtype=np.uint8).tobytes()
        elif kind == 1:
            s = rng.integers(97, 101, m, dtype=np.uint8).tobytes()
        elif kind == 2:
            s = bytes(m)
        else:
            s = b" ".join(words[int(k)] for k in rng.integers(0, len(words), m // 4 + 1))[:m]
        parts.append(s)
        total += len(s)
    return b"".join(parts)[:n]


def equality_pages(page: int, wm: int, seed: int = 0, port=None) -> dict:
    """{d: page bytes} with len(compress_fragment(page)) == page + d for d in (1, 0, -1): random bytes with a run of
    one byte value planted inside, the run's length searched.  Random bytes alone compress to page + 2 or 3; every
    byte of run saves about one.  (At 64 bytes d = +1 cannot occur: random bytes give +2 (a 64-byte literal has a
    2-byte header), and a copy of L >= 4 bytes costs 2 and a literal header, so a page with one comes to 4 - L or
    less.  Sizes below 64 are left out: every page of theirs is stored.)"""
    port = port or oracle.port()
    want = 2 if page == 64 else 3
    found = {}
    for s in range(64):
        rng = np.random.default_rng([seed, page, wm, s])
        base = bytearray(rng.integers(0, 256, page, dtype=np.uint8).tobytes())
        at = int(rng.integers(0, min(page - 8, 512)))
        v = int(rng.integers(0, 256))
        for r in range(0, min(page - at, 160)):
            p = bytes(base[:at]) + bytes([v]) * r + bytes(base[at + r:])
            d = len(port.compress_fragment(p, wm)) - page
            if d in (1, 0, -1) and d not in found:
                found[d] = p
            if d < -1:
                break
        if len(found) == want:
            return found
    return found


def short_tail(seed: int, n: int, snappy: bool = False) -> bytes:
    """A last page of n (1..31) bytes, which the writer stores (its fragment is longer): random bytes, or with
    `snappy` a raw Snappy literal of n - 1 bytes, which the reader then decodes to those n - 1 bytes."""
    b = np.random.default_rng([seed, n]).integers(0, 256, n, dtype=np.uint8).tobytes()
    return bytes([(n - 2) << 2]) + b[1:] if snappy and n >= 2 else b


def container_input(page: int, wm: int, seed: int, tail: int, pages: int = 24) -> tuple[bytes, dict]:
    """One input holding every page class for this page size: the equality pages (compressed size page + 1, page,
    page - 1), random (stored), zero and text pages, mixed pages, then a short last page of `tail` random bytes.
    -> (bytes, {class: [page indexes]})."""
    rng = np.random.default_rng([seed, page, wm])
    out, cls = [], {}

    def add(name, p):
        cls.setdefault(name, []).append(len(out))
        out.append(p)

    if page >= 64:
        for d, p in equality_pages(page, wm, seed).items():
            add(f"eq{d:+d}", p)
    for _ in range(3):
        add("random", rng.integers(0, 256, page, dtype=np.uint8).tobytes())
        add("zero", bytes(page))
        add("text", rng.integers(97, 100, page, dtype=np.uint8).tobytes())
    mixed = mixed_bytes(int(rng.integers(1 << 30)), page * pages, scale=max(page, 64))
    for i in range(pages):
        add("mixed", mixed[i * page:(i + 1) * page])
    data = b"".join(out)
    if tail:
        cls["short_tail"] = [len(out)]
        data += short_tail(seed, tail)
    return data, cls


CHUNK_MIN = 256  # the smallest chunk, which every input of up to 4 * 256 pages per worker gets


def edge_lengths(page: int, ks=(1, 2)) -> list[int]:
    """k * chunk * page + {-1, 0, 1, page - 1} for chunk = CHUNK_MIN: a last chunk that ends one byte early, is
    exactly full, holds one 1-byte page, or one page one byte short."""
    out = []
    for k in ks:
        for d in (-1, 0, 1, page - 1):
            n = k * CHUNK_MIN * page + d
            if n > 0 and n not in out:
                out.append(n)
    return out


# ------------------------------------------------------------------------------------------- hostile containers
@dataclass
class Hostile:
    name: str
    cls: str
    cont: bytes
    capacity_pages: int | None = None  # out capacity in pages (None: nr)


def _parse(cont: bytes):
    nr = struct.unpack_from("<I", cont, 0)[0]
    idx = list(np.frombuffer(cont, dtype="<u4", count=nr, offset=4).astype(np.int64))
    pos = 4 + 4 * nr
    payloads = []
    for cl in idx:
        payloads.append(cont[pos:pos + int(cl)])
        pos += int(cl)
    return payloads


def _build(payloads, idx=None) -> bytes:
    idx = [len(p) for p in payloads] if idx is None else idx
    return struct.pack("<I", len(idx)) + b"".join(struct.pack("<I", x) for x in idx) + b"".join(payloads)


_BAD_COPY = bytes([0xFE, 0xFF, 0xFF])  # copy-2 of 64 bytes at offset 65535, before anything was produced: -5


def hostile_containers(cont: bytes, page: int, chunk: int, seed: int) -> list[Hostile]:
    """Corruptions of a valid container (several chunks of `chunk` pages) in every class the reader treats apart.
    Payloads are rebuilt to match a changed entry where the class is about the entry, so the pages behind it stay
    in place."""
    rng = np.random.default_rng(seed)
    pay = _parse(cont)
    nr = len(pay)
    mc = max_clen(page)
    comp = [i for i, p in enumerate(pay) if 8 < len(p) < page]  # compressed pages
    assert nr >= 3 * chunk and len(comp) >= 8, (nr, chunk, len(comp))
    mid = nr // 2
    out = []

    def with_entry(i, cl):
        p = list(pay)
        src = pay[i] + rng.integers(0, 256, max(0, cl - len(pay[i])), dtype=np.uint8).tobytes()
        p[i] = src[:cl]
        return _build(p)

    for i in (0, mid, nr - 1):
        for cl, tag in ((0, "0"), (page - 1, "page-1"), (page, "page"), (page + 1, "page+1"), (mc, "max_clen"),
                        (mc + 1, "max_clen+1")):
            out.append(Hostile(f"entry {tag} at page {i}", f"entry_{tag}", with_entry(i, cl)))
    # a payload running past the end of the container, at page 0, in the middle, at a chunk's first page, at the last
    starts = np.cumsum([4 + 4 * nr] + [len(p) for p in pay])
    for i, tag in ((0, "first"), (mid, "middle"), (chunk, "chunk_first"), (2 * chunk, "chunk_first"), (nr - 1, "last")):
        if len(pay[i]):
            cut = int(starts[i] + len(pay[i]) - 1)
            out.append(Hostile(f"payload of page {i} past the end", f"past_end_{tag}", cont[:cut]))
    # decode failures in two different chunks (the later one first in the index order of no worker)
    a = next(i for i in comp if i >= chunk)
    b = next(i for i in comp if i >= 2 * chunk + chunk // 2)
    p = list(pay)
    p[a] = _BAD_COPY + pay[a][3:]
    p[b] = _BAD_COPY + pay[b][3:]
    out.append(Hostile(f"decode failures at pages {a} and {b}", "two_chunks", _build(p)))
    p = list(pay)
    p[b] = _BAD_COPY + pay[b][3:]
    out.append(Hostile(f"decode failure at page {b} only", "one_failure", _build(p)))
    # an index error before a decode error, and one after
    p = list(pay)
    p[b] = _BAD_COPY + pay[b][3:]
    idx = [len(x) for x in p]
    idx[a] = mc + 1
    out.append(Hostile(f"index error at {a} before decode error at {b}", "index_before_decode", _build(p, idx)))
    p = list(pay)
    p[a] = _BAD_COPY + pay[a][3:]
    idx = [len(x) for x in p]
    idx[b] = mc + 1
    out.append(Hostile(f"decode error at {a} before index error at {b}", "index_after_decode", _build(p, idx)))
    # a payload cut short inside the index scan's reach (a decode error that is -5 or -3 by the oracle), random bytes
    p = list(pay)
    c = comp[len(comp) // 3]
    p[c] = rng.integers(0, 256, len(pay[c]), dtype=np.uint8).tobytes()
    out.append(Hostile(f"random payload at page {c}", "random_payload", _build(p)))
    # header-level cases
    out.append(Hostile("nr = 0", "nr_0", struct.pack("<I", 0) + cont[4:]))
    out.append(Hostile("nr = 0xFFFFFFFF, short container", "nr_max", struct.pack("<I", 0xFFFFFFFF) + cont[4:]))
    out.append(Hostile("index cut inside", "short_index", cont[:4 + 4 * (nr - 1) + 2]))
    out.append(Hostile("capacity one byte below nr * page", "capacity", cont, capacity_pages=-1))
    return out


HOSTILE_CLASSES = {f"entry_{t}" for t in ("0", "page-1", "page", "page+1", "max_clen", "max_clen+1")} | {
    f"past_end_{t}" for t in ("first", "middle", "chunk_first", "last")} | {
    "two_chunks", "one_failure", "index_before_decode", "index_after_decode", "random_payload", "nr_0", "nr_max",
    "short_index", "capacity"}


def capacity_of(h: Hostile, nr: int, page: int) -> int:
    return nr * page - 1 if h.capacity_pages == -1 else nr * page
