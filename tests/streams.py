"""Snappy raw streams built tag by tag, with the decoder's result known by construction.

Stream appends literal and copy tags in any encoding the format allows -- copy-4 tags, copies of 1-3
bytes, 3- and 4-byte literal lengths, long-form lengths on short literals, the zero-length literal
`fc ff ff ff ff` -- none of which csnappy's own compressor writes.  It keeps the tags as a list, and
Stream.expect(cap, end) replays that list with the checks of csnappy_decompress_noheader, in the
reference's order:

  * a tag header cut off by the end of input is -5 (undefined in the reference, defined so here);
  * literal: payload shorter than its length -5, then no space -3 (a length of 2^31 or more skips the
    payload test and fails on space);
  * copy: offset 0 or beyond what was produced -5, then no space -3;
  * the end of input at a tag boundary is success.

The replay never parses the encoded bytes, so it is independent of every decoder it is compared with.

Generators (all seeded): copy_matrix, boundary_streams, random_stream / long_stream, invalid_cases and
overlong_streams.  A Case is a stream, a capacity and optionally an input length that cuts the stream.
"""
from __future__ import annotations

import numpy as np

NO_CAP = 0xFFFFFFFF
E_OK, E_OUTPUT_OVERRUN, E_DATA_MALFORMED = 0, -3, -5

SMALL_OFFSETS = tuple(range(1, 71)) + (127, 128, 2047, 2048)
LARGE_OFFSETS = (32767, 32768, 32769, 65535, 65536, 65537, 100000)
LARGE_LENGTHS = (1, 2, 3, 4, 7, 8, 9, 11, 15, 16, 17, 31, 32, 33, 63, 64)
PHASES = (0, 1, 7, 8, 9, 15)
LIT_LENGTHS = (1, 60, 61, 256, 257, 527, 528, 529, 65536, 65537)
COPY_HDR = {1: 2, 2: 3, 4: 5}


class Stream:
    def __init__(self):
        self.buf = bytearray()
        self.tags = []  # (start, header bytes, kind 0 literal / 1, 2, 4 copy, length, offset, payload)
        self.produced = 0  # output length if every tag so far is valid

    def lit(self, data: bytes, form: int | None = None, field: int | None = None):
        """Literal of `data` with `form` length bytes (0: length in the tag; 1-4: after it; None: the shortest).
        `field` overrides the stored length - 1 (a literal whose length differs from its payload ends the stream)."""
        n = len(data)
        field = n - 1 if field is None else field
        if form is None:
            form = 0 if field < 60 else (field.bit_length() + 7) // 8
        assert 0 <= field <= 0xFFFFFFFF and (field < 60 if form == 0 else 1 <= form <= 4 and field < 256 ** form)
        start = len(self.buf)
        if form == 0:
            self.buf.append(field << 2)
        else:
            self.buf.append((59 + form) << 2)
            self.buf += field.to_bytes(form, "little")
        length = (field + 1) & 0xFFFFFFFF
        self.tags.append((start, 1 + form, 0, length, 0, bytes(data)))
        self.buf += data
        self.produced += length
        return self

    def zero_lit(self):
        """`fc ff ff ff ff`: the 4-byte length 0xffffffff + 1 wraps to an empty literal."""
        return self.lit(b"", form=4, field=0xFFFFFFFF)

    def copy(self, off: int, n: int, kind: int | None = None):
        """Copy of n bytes from `off` back with a copy-1 / copy-2 / copy-4 tag (None: the shortest)."""
        if kind is None:
            kind = 1 if 4 <= n <= 11 and off < 2048 else (2 if off < 65536 else 4)
        if kind == 1:
            assert 4 <= n <= 11 and 0 <= off < 2048
            tag = 1 | ((n - 4) << 2) | ((off >> 8) << 5)
            enc = bytes([tag, off & 0xFF])
        else:
            assert 1 <= n <= 64 and 0 <= off < (1 << (8 * kind))
            enc = bytes([(2 if kind == 2 else 3) | ((n - 1) << 2)]) + off.to_bytes(kind, "little")
        self.tags.append((len(self.buf), COPY_HDR[kind], kind, n, off, b""))
        self.buf += enc
        self.produced += n
        return self

    def pad_to(self, pos: int, rng):
        """Short literals until the stream is exactly `pos` bytes long (pos - len >= 2)."""
        d = pos - len(self.buf)
        assert d >= 2 or d == 0
        while d:
            t = min(d, 61)
            if d - t == 1:
                t -= 1
            self.lit(rng.bytes(t - 1))
            d -= t
        return self

    def expect(self, cap: int = NO_CAP, end: int | None = None):
        """-> (rc, index of the failing tag or None, produced bytes or None) of decoding buf[:end] into `cap` bytes."""
        end = len(self.buf) if end is None else end
        out = bytearray()
        for i, (start, hdr, kind, length, off, payload) in enumerate(self.tags):
            if start >= end:
                break
            room = cap - len(out)
            if end - start < hdr:
                return E_DATA_MALFORMED, i, None
            if kind == 0:
                avail = min(end, len(self.buf)) - start - hdr
                if length < 1 << 31:
                    if avail < length:
                        return E_DATA_MALFORMED, i, None
                    assert length == len(payload), "a literal longer than its payload must end the stream"
                elif room >= length:  # the reference's signed test, reachable only with a capacity of 2 GiB or more
                    return E_DATA_MALFORMED, i, None
                if room < length:
                    return E_OUTPUT_OVERRUN, i, None
                out += payload
            else:
                if off == 0 or off > len(out):
                    return E_DATA_MALFORMED, i, None
                if room < length:
                    return E_OUTPUT_OVERRUN, i, None
                src = out[len(out) - off: len(out) - off + length]
                if off < length:  # overlapping: the last `off` bytes repeat
                    src = (src * (length // off + 1))[:length]
                out += src
        return E_OK, None, bytes(out)

    def with_header(self, n: int | None = None) -> bytes:
        """buf behind a varint32 length (csnappy_decompress's format); n defaults to the produced length."""
        n = self.produced if n is None else n
        h = bytearray()
        while n >= 128:
            h.append((n & 0x7F) | 0x80)
            n >>= 7
        h.append(n)
        return bytes(h) + bytes(self.buf)


class Case:
    """A stream decoded into `cap` bytes, optionally cut to its first `end` input bytes."""

    def __init__(self, s: Stream, cap: int | None = None, end: int | None = None, name: str = ""):
        self.s, self.end, self.name = s, end, name
        self.cap = s.produced if cap is None else cap
        assert 0 <= self.cap <= NO_CAP
        self.data = bytes(s.buf[:end]) if end is not None else bytes(s.buf)
        self._exp = {}

    def expect(self, cap: int | None = None):
        cap = self.cap if cap is None else cap
        if cap not in self._exp:
            self._exp[cap] = self.s.expect(cap, self.end)
        return self._exp[cap]


# ---- (a) every copy form at every offset class, length and output phase ----------------------------------
def copy_matrix(seed: int, kinds=(1, 2, 4), offsets=SMALL_OFFSETS, lengths=None, phases=PHASES):
    """One stream per (kind, offset, length, phase): random literal bytes that end at output phase `phase`
    (mod 16) and reach back at least `offset`, the copy, the same copy again, a short literal."""
    rng = np.random.default_rng(seed)
    cases = []
    for kind in kinds:
        lim = {1: 2048, 2: 65536, 4: 1 << 32}[kind]
        for off in offsets:
            if off >= lim:
                continue
            for n in (lengths or (range(4, 12) if kind == 1 else range(1, 65))):
                if kind == 1 and not 4 <= n <= 11:
                    continue
                for ph in phases:
                    p = off + (ph - off) % 16
                    s = Stream().lit(rng.bytes(p)).copy(off, n, kind).copy(off, n, kind)
                    s.lit(rng.bytes(int(rng.integers(1, 17))))
                    cases.append(Case(s, name=f"copy{kind} off {off} len {n} phase {ph}"))
    return cases


def large_copy_matrix(seed: int):
    return copy_matrix(seed, kinds=(2, 4), offsets=LARGE_OFFSETS, lengths=LARGE_LENGTHS, phases=(0, 7, 15))


# ---- (b) sequences at the decoders' boundaries ------------------------------------------------------------
def boundary_streams(seed: int):
    rng = np.random.default_rng(seed)
    cases = []
    # every literal length class in every length form that holds it, at three output phases, then a copy
    for n in LIT_LENGTHS:
        for form in range(5):
            if (form == 0 and n > 60) or (form and n - 1 >= 256 ** form):
                continue
            for ph in (0, 1, 7):
                s = Stream()
                if ph:
                    s.lit(rng.bytes(ph))
                s.lit(rng.bytes(n), form=form).copy(min(n + ph, 40), 20, 2).lit(rng.bytes(5))
                cases.append(Case(s, name=f"literal {n} form {form} phase {ph}"))
    # the zero-length literal between, before and after other tags
    s = Stream().zero_lit().lit(rng.bytes(30)).zero_lit().zero_lit().copy(7, 50, 2).zero_lit()
    cases.append(Case(s, name="zero-length literals"))
    # pattern runs longer than 256 bytes: the same offset over many tags, every offset class
    for off in (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 30, 31, 32, 33, 63):
        for kind in (2, 4):
            s = Stream().lit(rng.bytes(off + 3))
            for n in (64, 64, 64, 64, 33, 64, 17, 64, 1, 64, 2, 3, 64):
                s.copy(off, n, kind)
            s.lit(rng.bytes(9))
            cases.append(Case(s, name=f"pattern run off {off} copy{kind}"))
    # runs of G and G/2 short tags with a long literal / a dependent copy / an overlapping copy at every position,
    # so that batches (G tags staged, G/2 global) and steps (G/8 tags) split everywhere
    for ntags in (4, 8, 16, 32, 33, 64):
        for j in range(ntags):
            for special in ("longlit", "dep", "overlap"):
                s = Stream().lit(rng.bytes(40))
                for t in range(ntags):
                    if t == j and special == "longlit":
                        s.lit(rng.bytes(int(rng.integers(61, 200))))
                    elif t == j and special == "dep":
                        # source ends inside the output of the tag just before (a literal of 12 bytes)
                        s.lit(rng.bytes(12)).copy(16, 10, 2)
                    elif t == j:
                        s.copy(3, 40, 4)
                    elif t % 3 == 0:
                        s.lit(rng.bytes(int(rng.integers(1, 9))))
                    else:
                        s.copy(int(rng.integers(8, 40)), int(rng.integers(1, 9)), 2 if t % 3 == 1 else 4)
                cases.append(Case(s, name=f"{ntags} tags, {special} at {j}"))
    # every step position: dependent copies (source in the previous tag's output, offset >= length) in a row
    for lead in range(8):
        s = Stream().lit(rng.bytes(24))
        for _ in range(lead):
            s.copy(24, 4, 1)
        for _ in range(12):
            s.lit(rng.bytes(6)).copy(8, 5, 2).copy(7, 7, 1).copy(12, 3, 4)
        cases.append(Case(s, name=f"dependent chain after {lead}"))
    return cases


# ---- (c) random valid streams -----------------------------------------------------------------------------
def _random_tag(s: Stream, rng, long_lits: bool = True):
    r = rng.random()
    p = s.produced
    if p == 0 or r < 0.25:
        n = int(rng.integers(61, 3000)) if long_lits and rng.random() < 0.1 else int(rng.integers(1, 61))
        forms = [f for f in range(5) if (n <= 60 if f == 0 else n - 1 < 256 ** f)]
        s.lit(rng.bytes(n), form=None if rng.random() < 0.8 else int(rng.choice(forms)))
    elif r < 0.27:
        s.zero_lit()
    else:
        kind = int(rng.choice([1, 2, 4]))
        far = rng.random() < 0.3
        lim = min(p, {1: 2047, 2: 65535, 4: p}[kind])
        off = int(rng.integers(1, lim + 1)) if far else int(rng.integers(1, min(lim, 70) + 1))
        n = int(rng.integers(4, 12)) if kind == 1 else int(rng.integers(1, 65))
        s.copy(off, n, kind)


def random_stream(seed: int, out_len: int) -> Stream:
    """Random tags of every form until at least out_len bytes are produced."""
    rng = np.random.default_rng(seed)
    s = Stream()
    while s.produced < out_len:
        _random_tag(s, rng)
    return s


# header sizes 2, 3, 4 and 5 in every encoding, for the input-chunk-edge placements of long_stream
_EDGE_TAGS = ("copy1", "copy2", "copy4", "lit1", "lit2", "lit3", "zero")


def _edge_tag(s: Stream, what: str, rng):
    p = s.produced
    if what == "copy1":
        s.copy(int(rng.integers(1, min(p, 2047) + 1)), 7, 1)
    elif what == "copy2":
        s.copy(int(rng.integers(256, min(p, 65535) + 1)), 9, 2)
    elif what == "copy4":  # offset bytes 3 and 4 in use whenever the output allows
        s.copy(int(rng.integers(min(p, 65536), p + 1)), 11, 4)
    elif what == "lit1":
        s.lit(rng.bytes(int(rng.integers(61, 256))), form=1)
    elif what == "lit2":
        s.lit(rng.bytes(int(rng.integers(256, 4000))), form=2)
    elif what == "lit3":
        s.lit(rng.bytes(65536 + int(rng.integers(1, 500))), form=3)
    else:
        s.zero_lit()


def long_stream(seed: int, out_len: int, chunk: int = 4096) -> Stream:
    """A random stream of at least out_len bytes that also has: copy-4 offsets spread over the whole output, an
    offset-1 run of more than 1 MiB (when out_len allows), literals over several input chunks, and tag headers of
    2, 3, 4 and 5 bytes placed so that each of their bytes in turn is the last one before an input position that is
    a multiple of `chunk`."""
    rng = np.random.default_rng(seed)
    s = Stream()
    s.lit(rng.bytes(3000))
    edges = [(w, j) for w in _EDGE_TAGS for j in range({"copy1": 2, "copy2": 3, "copy4": 5, "lit1": 2, "lit2": 3,
                                                         "lit3": 4, "zero": 5}[w])]
    if out_len >= 4 << 20:
        edges += edges  # a second round further into the stream
    run_at = out_len // 3 if out_len >= 3 << 20 else None
    step = max(1, out_len // (len(edges) + 2))
    next_edge = step
    while s.produced < out_len:
        if run_at is not None and s.produced >= run_at:
            s.lit(rng.bytes(1))
            for _ in range((1 << 20) // 64 + 2):
                s.copy(1, 64, int(rng.choice([2, 4])))
            run_at = None
        elif edges and s.produced >= next_edge and s.produced > 70000:
            what, j = edges.pop(0)
            target = (len(s.buf) // chunk + 1) * chunk - 1 - j
            if target - len(s.buf) < 2:
                target += chunk
            s.pad_to(target, rng)
            _edge_tag(s, what, rng)
            next_edge += step
        elif rng.random() < 0.001:
            s.lit(rng.bytes(int(rng.integers(4 * chunk, 12 * chunk))))  # over several input chunks
        elif rng.random() < 0.05 and s.produced > 65536:
            s.copy(int(rng.integers(65536, s.produced + 1)), int(rng.integers(1, 65)), 4)
        else:
            _random_tag(s, rng)
    return s


def stream_of_input_len(seed: int, src_len: int) -> Stream:
    """A random valid stream of exactly src_len input bytes (src_len >= 2)."""
    rng = np.random.default_rng(seed)
    s = Stream()
    while src_len - len(s.buf) >= 70:  # a short tag is at most 65 bytes: at least 5 are left to pad
        _random_tag(s, rng, long_lits=False)
    return s.pad_to(src_len, rng)


# ---- (d) invalid streams ----------------------------------------------------------------------------------
def invalid_cases(seed: int):
    rng = np.random.default_rng(seed)
    cases = []

    def base(n):
        return random_stream(int(rng.integers(1 << 30)), n)

    for k in range(24):
        n = int(rng.integers(100, 3000))
        # bad offsets, followed by more valid-looking tags
        for off_of, kind in ((lambda p: 0, 2), (lambda p: p + 1, 1), (lambda p: p + 1, 2), (lambda p: p + 1, 4),
                             (lambda p: 0xFFFFFFFF, 4), (lambda p: 0, 4)):
            s = base(n)
            p = s.produced
            if kind == 1 and p + 1 >= 2048:
                continue
            s.copy(off_of(p), 5, kind).lit(rng.bytes(10)).copy(1, 8, 2)
            cases.append(Case(s, name="bad offset"))
        # copy-4 offsets whose upper bytes matter: the low 16 / 24 bits alone would be a valid offset
        for hi in (1 << 16, 1 << 24, 0x5A << 24):
            s = base(n)
            s.copy(hi + int(rng.integers(1, 40)), 6, 4).lit(rng.bytes(4))
            cases.append(Case(s, name="copy-4 offset above 16 bits"))
        # capacities around what is needed
        s = base(n)
        for d in (-1, 0, 1):
            cases.append(Case(s, cap=s.produced + d, name=f"cap needed{d:+d}"))
        cases.append(Case(s, cap=int(rng.integers(0, s.produced)), name="cap short"))
        # a literal length of 2^31 or more: fails on space
        for field in ((1 << 31) - 1, 0xFFFFFFFE, (1 << 31) + 12345):
            s = base(n)
            p = s.produced
            s.lit(rng.bytes(20), form=4, field=field)
            cases.append(Case(s, cap=p + 100, name="literal length >= 2^31"))
        # the header of each tag kind cut at each byte, and a literal payload one byte short
        for what in ("copy1", "copy2", "copy4", "lit1", "lit2", "lit3", "lit4"):
            s = base(n)
            if what.startswith("copy"):
                s.copy(int(rng.integers(1, 100)), 8, int(what[4]))
            else:
                s.lit(rng.bytes(int(rng.integers(1, 257))), form=int(what[3]))
            start, hdr = s.tags[-1][:2]
            for j in range(hdr + 1):
                cases.append(Case(s, end=start + j, name=f"{what} header cut at {j}"))
            if what.startswith("lit"):
                cases.append(Case(s, end=len(s.buf) - 1, name="literal payload one byte short"))
        # two errors in one tag: the first check in the reference's order wins
        s = base(n)
        p = s.produced
        s.lit(rng.bytes(50), form=2, field=99)  # payload short by 50 bytes
        cases.append(Case(s, cap=p + 10, name="literal short and no space"))
        s = base(n)
        p = s.produced
        s.copy(p + 1, 30, 2)
        cases.append(Case(s, cap=p + 3, name="bad offset and no space"))
        # an invalid tag behind a valid tag that does not fit: the earlier failure decides
        s = base(n)
        p = s.produced
        s.lit(rng.bytes(20)).copy(p + 100, 4, 4)
        cases.append(Case(s, cap=p + 5, name="no space before a bad offset"))
    return cases


# ---- (e) inputs longer than max_compressed_length(cap) -----------------------------------------------------
def overlong_streams(seed: int, sizes=(1000, 4096, 32768)):
    """Streams of 1-byte literals (2 input bytes per output byte) and streams padded with zero-length literals;
    valid, and with capacity one short."""
    rng = np.random.default_rng(seed)
    cases = []
    for n in sizes:
        s = Stream()
        data = rng.bytes(n)
        for i in range(n):
            s.lit(data[i:i + 1])
        cases += [Case(s, name=f"{n} 1-byte literals"), Case(s, cap=n - 1, name=f"{n} 1-byte literals, cap - 1")]
        s = Stream()
        while s.produced < n:
            s.zero_lit()
            if rng.random() < 0.2:
                _random_tag(s, rng)
        cases += [Case(s, name=f"{n} zero-length padding"), Case(s, cap=s.produced - 1, name="padding, cap - 1")]
    return cases
