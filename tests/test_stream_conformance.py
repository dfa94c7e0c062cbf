"""The CPU oracle port against streams whose result is known by construction (tests/streams.py).

The port (oracle/snappy_oracle.c) is the reference the GPU decoder tests compare with, but until now it was
only checked on what csnappy's compressor writes and on corruptions of that.  Here it decodes every tag
form of the format -- copy-4 tags, copies of 1-3 bytes, literals with 1-4 length bytes on any length, the
zero-length literal, offsets up to 2^32 - 1 -- valid and invalid, and its return code and bytes must equal
the replay of the stream's tag list.  The GPU file tests/test_gpu_decode_conformance.py relies on this.
"""
import functools
import os
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle  # noqa: E402
import streams as S  # noqa: E402


@functools.lru_cache(maxsize=None)
def all_cases():
    cases = (S.copy_matrix(101) + S.large_copy_matrix(102) + S.boundary_streams(103) + S.invalid_cases(104) +
             S.overlong_streams(105))
    for seed, n in ((1, 4096), (2, 32768), (3, 1 << 20)):
        cases.append(S.Case(S.random_stream(seed, n), name=f"random {n}"))
    s = S.long_stream(4, 3 << 20)
    cases += [S.Case(s, name="long"), S.Case(s, cap=s.produced - 1, name="long, cap - 1"),
              S.Case(s, end=len(s.buf) * 2 // 3, name="long, cut")]
    for n in (1, 4095, 4096, 4097):
        cases.append(S.Case(S.stream_of_input_len(n, max(n, 2)), name=f"{n} input bytes"))
    return cases


def test_port_decodes_every_stream_as_constructed():
    port = oracle.port()
    n_err = 0
    for c in all_cases():
        rc, _, out = c.expect()
        got_rc, got = port.decompress_noheader(c.data, c.cap)
        assert got_rc == rc, (c.name, c.cap, c.data[:40].hex())
        if rc == 0:
            assert got == out, c.name
        else:
            n_err += 1
    assert n_err > 800


def test_port_decodes_the_header_form():
    """csnappy_decompress: varint32 length, -1 for a bad header, -2 when it is larger than the buffer, then the
    stream decoded into exactly the length the header states."""
    port = oracle.port()
    for c in all_cases()[::7]:
        if c.end is not None or c.s.produced > S.NO_CAP:
            continue
        n = c.s.produced
        rc, _, out = c.s.expect(n)
        got_rc, got = port.decompress(c.s.with_header(), n)
        assert got_rc == rc, c.name
        if rc == 0:
            assert got == out, c.name
        if n:
            assert port.decompress(c.s.with_header(), n - 1)[0] == oracle.E_OUTPUT_INSUF
    assert port.decompress(b"", 10)[0] == oracle.E_HEADER_BAD
    assert port.decompress(b"\xff\xff\xff\xff\xff\x00", 10)[0] == oracle.E_HEADER_BAD
    assert port.decompress(b"\x80\x80", 10)[0] == oracle.E_HEADER_BAD


def test_generators_cover_every_tag_form():
    kinds, lit_forms, short_copies, far, zero = set(), set(), set(), False, False
    rcs = set()
    for c in all_cases():
        for start, hdr, kind, length, off, _ in c.s.tags:
            kinds.add(kind)
            if kind == 0:
                lit_forms.add(hdr - 1)
                zero = zero or length == 0
            else:
                if length <= 3:
                    short_copies.add((kind, length))
                far = far or off > 65535
        rcs.add(c.expect()[0])
    assert kinds == {0, 1, 2, 4}
    assert lit_forms == {0, 1, 2, 3, 4}
    assert short_copies == {(k, n) for k in (2, 4) for n in (1, 2, 3)}
    assert far and zero
    assert rcs == {S.E_OK, S.E_OUTPUT_OVERRUN, S.E_DATA_MALFORMED}


@pytest.mark.parametrize("form", [1, 2, 3, 4])
def test_long_form_lengths_on_short_literals(form):
    """A 1-byte literal with every length form is the same literal."""
    s = S.Stream().lit(b"a", form=form).lit(b"bc", form=0).copy(3, 3, 2)
    assert s.expect() == (S.E_OK, None, b"abcabc")
    assert oracle.port().decompress_noheader(bytes(s.buf), 6) == (0, b"abcabc")
