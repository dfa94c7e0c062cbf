"""Streams placed on the parallel stream decoder's 4096-byte input chunks, with results known by construction.

stream_kernel.cu cuts its input into 4096-byte chunks: it ranks the speculative tag list inside each chunk, one
thread hops from chunk to chunk, and every chunk expands its own tags from where the real chain enters it.  A
stream from tests/streams.py meets that grid wherever its bytes happen to fall.  Two tools here put them where the
kernel can go wrong:

  * shifted(case, k) puts k zero-length literals (`fc ff ff ff ff`) in front of a case.  They add 5 input bytes each
    and no output, so offsets, capacities and the result stay what they were, and the failing tag's index moves by k.
    Because gcd(5, 4096) = 1, k_before(pos) (at most 4095, a prefix of at most 20 475 bytes) makes original byte
    `pos` the first byte of a chunk: a chunk boundary can be put before any byte of any case.
  * chunk_cases(seed) builds streams whose chunk structure is chosen: literals over whole chunks, a chunk entered at
    its last byte, a chunk of 2048 copy-1 tags with a failure at chosen tag indices, failures in different chunks,
    inputs of one byte around whole chunks.

big_literal_cases(seed) gives the literals of 2^31 bytes or more at capacities of 2 GiB and above, the only inputs
on which the reference's signed payload test makes a difference.
"""
from __future__ import annotations

import numpy as np

import streams as S

CHUNK = 4096
INV5 = pow(5, -1, CHUNK)  # 3277
ZERO_LIT = b"\xfc\xff\xff\xff\xff"
BIG_CAPS = ((1 << 31) + (1 << 20), S.NO_CAP)
BIG_FIELDS = ((1 << 31) - 1, 0xFFFFFFFE, (1 << 31) + 12345)


def shifted(case: S.Case, k: int) -> S.Case:
    """`case` behind k zero-length literals: the stream is rebuilt by replaying its tag list (literals keep their
    length form and field), a cut `end` moves by 5k, the capacity stays."""
    s = S.Stream()
    s.buf += ZERO_LIT * k
    s.tags = [(5 * i, 5, 0, 0, 0, b"") for i in range(k)]
    for start, hdr, kind, length, off, payload in case.s.tags:
        if kind == 0:
            s.lit(payload, form=hdr - 1, field=(length - 1) & 0xFFFFFFFF)
        else:
            s.copy(off, length, kind)
    end = None if case.end is None else case.end + 5 * k
    return S.Case(s, cap=case.cap, end=end, name=f"{case.name} +{k} zero literals")


def k_before(pos: int) -> int:
    """Zero-length literals that put byte `pos` of a stream at the start of a chunk (byte pos - 1 at offset 4095)."""
    return (-pos * INV5) % CHUNK


def failing_tag(case: S.Case) -> int:
    """Index of the tag that decides the result: the failing one, or the last one of a valid case."""
    _, i, _ = case.expect()
    return len(case.s.tags) - 1 if i is None else i


def header_shifts(case: S.Case):
    """Shifts that put a chunk boundary before each byte of the deciding tag's header and right after it."""
    start, hdr = case.s.tags[failing_tag(case)][:2]
    return [k_before(start + j) for j in range(hdr + 1)]


def last_tag_shifts(case: S.Case, payload: bool = True):
    """A chunk boundary before the last tag, inside its header (after its first byte) and inside its payload."""
    start, hdr, _, _, _, data = case.s.tags[-1]
    at = [start, start + max(1, hdr // 2)]
    if payload:
        at.append(start + hdr + max(1, len(data) // 2))
    return [k_before(p) for p in at]


def shift_plan():
    """(case, k) pairs of the shifted corpus, by part: every invalid case with a boundary before each byte of its
    deciding tag's header and after it; the boundary, large-copy and overlong streams with a boundary before, inside
    the header of and inside the payload of their last tag; every 8th copy-matrix stream before and inside the header
    of its last tag.  The seeds are those of test_gpu_decode_conformance.py."""
    edges = S.boundary_streams(203) + S.large_copy_matrix(202) + S.overlong_streams(205)
    return {
        "invalid": [(c, k) for c in S.invalid_cases(204) for k in header_shifts(c)],
        "edges": [(c, k) for c in edges for k in last_tag_shifts(c)],
        "copy_matrix": [(c, k) for c in S.copy_matrix(201)[::8] for k in last_tag_shifts(c, payload=False)],
    }


# ---- streams with a chosen chunk structure ----------------------------------------------------------------
def _lit_to(s: S.Stream, last: int, rng, form: int = 3):
    """A literal with a `form`-byte length that starts at the end of s and whose last payload byte is at `last`."""
    n = last + 1 - len(s.buf) - 1 - form
    assert n >= 1
    return s.lit(rng.bytes(n), form=form)


def _near_copy(s: S.Stream, rng, kind: int = 2):
    n = int(rng.integers(4, 12)) if kind == 1 else int(rng.integers(1, 65))
    return s.copy(int(rng.integers(1, min(s.produced, 2047) + 1)), n, kind)


def chunk_cases(seed: int):
    rng = np.random.default_rng(seed)
    cases = []

    # a literal over two or more whole chunks whose last byte is at offset 4095, 0 or 1 of a chunk, then a valid copy
    # or a bad offset: every chunk it covers has no chain entry
    for last_off in (4095, 0, 1):
        for tail in ("copy", "bad offset"):
            s = S.Stream().lit(rng.bytes(100)).pad_to(1000, rng)
            _lit_to(s, 4 * CHUNK + last_off if last_off != 4095 else 3 * CHUNK + last_off, rng)
            if tail == "copy":
                s.copy(int(rng.integers(1, 5000)), 40, 2)
            else:
                s.copy(s.produced + 1, 40, 2)
            s.lit(rng.bytes(7)).copy(3, 9, 1)
            cases.append(S.Case(s, name=f"literal over whole chunks ending at offset {last_off}, {tail}"))

    # a chunk entered at its last byte: a literal ends at offset 4094, a copy-1 tag starts at 4095
    for what in ("valid", "bad offset", "no space"):
        s = S.Stream().lit(rng.bytes(3000))
        _lit_to(s, 2 * CHUNK + 4094, rng, form=2)
        p = s.produced
        s.copy(0 if what == "bad offset" else 1000, 7, 1)
        for _ in range(20):
            _near_copy(s, rng, 1)
        s.lit(rng.bytes(3))
        assert s.tags[-22][0] == 2 * CHUNK + 4095
        cases.append(S.Case(s, cap=p + 6 if what == "no space" else None, name=f"chunk entered at offset 4095, {what}"))

    # a chunk of 2048 copy-1 tags (its tag list and 32-entry spine full), a failing tag at index t of the chunk
    for t in (None, 0, 63, 64, 65, 2047):
        for what in (("bad offset", "no space") if t is not None else ("valid",)):
            s = S.Stream().lit(rng.bytes(2500)).pad_to(2 * CHUNK, rng)
            first = len(s.tags)
            cap = None
            for i in range(2048):
                if i == t and what == "bad offset":
                    s.copy(0, 5, 1)
                else:
                    if i == t:
                        cap = s.produced + 3
                    _near_copy(s, rng, 1)
            assert len(s.buf) == 3 * CHUNK and s.tags[first][0] == 2 * CHUNK
            s.lit(rng.bytes(30)).copy(30, 64, 2)
            at = "" if t is None else f" at tag {t}"
            cases.append(S.Case(s, cap=cap, name=f"2048 copy-1 tags, {what}{at}"))

    # two failures in different chunks: the smaller position wins whatever its class
    for order in ("-3 then -5", "-5 then -3"):
        s = S.Stream().lit(rng.bytes(3000)).pad_to(CHUNK + 100, rng)
        if order == "-3 then -5":
            cap = s.produced + 10
            s.copy(50, 20, 2)
        else:
            s.copy(0, 20, 2)
        s.pad_to(3 * CHUNK + 200, rng)
        if order == "-3 then -5":
            s.copy(s.produced + 1, 20, 4)
        else:
            cap = s.produced + 10
            s.copy(50, 20, 4)
        s.lit(rng.bytes(9))
        cases.append(S.Case(s, cap=cap, name=f"failures in chunks 1 and 3, {order}"))

    # a non-terminal failure before a terminal header cut at the end of the input
    for what in ("bad offset", "no space"):
        s = S.Stream().lit(rng.bytes(2000)).pad_to(CHUNK - 300, rng)
        cap = s.produced + 5 if what == "no space" else None
        s.copy(0 if what == "bad offset" else 10, 30, 2)
        s.pad_to(2 * CHUNK + 50, rng)
        s.copy(100, 10, 4)
        cases.append(S.Case(s, cap=cap, end=len(s.buf) - 2, name=f"{what} before a terminal header cut"))

    # inputs of one byte around whole chunks, with the capacity needed and one byte less; the same lengths again
    # with a last literal across the last chunk boundary below the end
    for k in (1, 2, 5):
        for n in (k * CHUNK - 1, k * CHUNK, k * CHUNK + 1):
            s = S.stream_of_input_len(1000 * k + n % 7, n)
            cases += [S.Case(s, name=f"{n} input bytes"), S.Case(s, cap=s.produced - 1, name=f"{n} input bytes, cap - 1")]
            b = (n - 1) // CHUNK * CHUNK
            if b == 0:
                continue
            s = S.Stream().lit(rng.bytes(200)).pad_to(b - 300, rng)
            _near_copy(s, rng, 4)
            s.pad_to(b - 3, rng)
            _lit_to(s, n - 1, rng, form=0 if n - b <= 58 else 2)
            assert len(s.buf) == n and s.tags[-1][0] < b <= n - 1
            cases += [S.Case(s, name=f"{n} input bytes, last literal across {b}"),
                      S.Case(s, cap=s.produced - 1, name=f"{n} input bytes, last literal across {b}, cap - 1")]
    return cases


# ---- literals of 2^31 bytes or more at capacities of 2 GiB and above --------------------------------------
def big_literal_cases(seed: int):
    """A short valid prefix, then a literal whose length field is 0x7fffffff, 0xfffffffe or 0x80003039, at
    capacities p + 100, 2^31 + 2^20 and 2^32 - 1.  The length is 2^31 or more, so the reference skips its payload
    test and fails on space; with room for the length the result is -5."""
    rng = np.random.default_rng(seed)
    cases = []
    for field in BIG_FIELDS:
        s = S.random_stream(int(rng.integers(1 << 30)), 300)
        p = s.produced
        s.lit(rng.bytes(20), form=4, field=field)
        for cap in (p + 100,) + BIG_CAPS:
            cases.append(S.Case(s, cap=cap, name=f"literal field {field:#x}, cap {cap:#x}"))
    return cases


# ---- outputs above 2^31 and running output offsets above 2^32 (too many tags for Stream: built with numpy) -----
RUN_TAG = b"\xfe\x01\x00"  # copy-2, length 64, offset 1


def _copy4(off: int, n: int) -> bytes:
    return bytes([3 | ((n - 1) << 2)]) + off.to_bytes(4, "little")


class RunStream:
    """A 4096-byte random literal, `fe 01 00` until at least `run_to` bytes are produced, copy-4 tags whose offsets
    reach back over the whole run into the first literal, and a short literal.  The output is known in pieces:
    head, head[-1] repeated up to run_end, head[x:x + n] at each (o, x, n) of `copies`, then `tail`."""

    def __init__(self, seed: int, run_to: int, n_copies: int = 24):
        rng = np.random.default_rng(seed)
        self.head = rng.bytes(CHUNK)
        runs = -(-(run_to - CHUNK) // 64)
        self.run_end = CHUNK + 64 * runs
        parts = [b"\xf4\xff\x0f", self.head, RUN_TAG * runs]
        o = self.run_end
        self.copies = []
        for _ in range(n_copies):
            n = int(rng.integers(1, 65))
            x = int(rng.integers(0, CHUNK - n + 1))
            parts.append(_copy4(o - x, n))
            self.copies.append((o, x, n))
            o += n
        self.tail = rng.bytes(11)
        parts += [bytes([(len(self.tail) - 1) << 2]), self.tail]
        self.data = b"".join(parts)
        self.produced = o + len(self.tail)

    def bad_offset_tail(self) -> bytes:
        """A copy-4 whose offset is one more than what was produced: appended to data, the stream fails with -5."""
        return _copy4(self.produced + 1, 8)


def saturating_stream(seed: int):
    """-> (input, cap): a literal, then a copy that does not fit `cap`, then `fe 01 00` tags until the running output
    offset passes 2^32 (the stream decoder saturates it), then a literal.  The result is -3."""
    rng = np.random.default_rng(seed)
    runs = (1 << 32) // 64 + 1000
    data = b"".join([b"\xf4\xff\x0f", rng.bytes(CHUNK), _copy4(1000, 64), RUN_TAG * runs, b"\x1c", rng.bytes(8)])
    return data, CHUNK + 63
