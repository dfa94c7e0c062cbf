"""The chunk-placed streams of tests/stream_chunks.py on the CPU: the shifted corpus keeps its construction result,
the boundaries land where they are meant to, the generators hold every structure they claim, and the CPU oracle
port decodes them as constructed.  test_gpu_stream_conformance.py relies on all of this: it sends the shifted bytes
through the stream decoder and compares with the unshifted expectation.
"""
import functools
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import oracle  # noqa: E402
import stream_chunks as C  # noqa: E402
import streams as S  # noqa: E402


@functools.lru_cache(maxsize=None)
def plan():
    return C.shift_plan()


def _check_shifts(pairs):
    for c, k in pairs:
        rc, i, out = c.expect()
        sc = C.shifted(c, k)
        assert sc.data == C.ZERO_LIT * k + c.data, c.name
        assert sc.expect() == (rc, None if i is None else i + k, out), (c.name, k)


def test_shifted_invalid_cases_keep_their_result():
    _check_shifts(plan()["invalid"])


def test_shifted_edge_streams_keep_their_result():
    _check_shifts(plan()["edges"])


def test_shifted_copy_matrix_keeps_its_result():
    _check_shifts(plan()["copy_matrix"])


def test_shifts_put_every_header_byte_at_the_end_of_a_chunk():
    """For every invalid case, the boundary falls before each byte of the deciding tag's header and right after it:
    each header byte is once at offset 4095 of a chunk."""
    assert len(plan()["invalid"]) == 6141
    for c in S.invalid_cases(204):
        start, hdr = c.s.tags[C.failing_tag(c)][:2]
        ks = C.header_shifts(c)
        assert len(ks) == hdr + 1 and max(ks) < C.CHUNK
        for j, k in enumerate(ks):
            assert (5 * k + start + j) % C.CHUNK == 0, c.name  # byte start + j opens a chunk
        assert {(5 * k + start + j - 1) % C.CHUNK for j, k in enumerate(ks[1:], 1)} == {C.CHUNK - 1}


def test_last_tag_shifts_land_before_inside_and_after_the_header():
    for c in S.boundary_streams(203) + S.overlong_streams(205):
        start, hdr, _, _, _, payload = c.s.tags[-1]
        at = [start, start + max(1, hdr // 2), start + hdr + max(1, len(payload) // 2)]
        ks = C.last_tag_shifts(c)
        assert [(5 * k + p) % C.CHUNK for k, p in zip(ks, at)] == [0, 0, 0]
        assert at[1] - start < hdr or hdr == 1
        assert at[2] < start + hdr + len(payload) or len(payload) <= 1


def test_chunk_cases_hold_every_structure():
    cases = C.chunk_cases(301)
    names = [c.name for c in cases]
    for last in (4095, 0, 1):
        for tail in ("copy", "bad offset"):
            c = cases[names.index(f"literal over whole chunks ending at offset {last}, {tail}")]
            lits = [(st + h, n) for st, h, kind, n, _, _ in c.s.tags if kind == 0 and n >= 2 * C.CHUNK]
            (p, n), = lits
            assert (p + n - 1) % C.CHUNK == last and (p + n - 1) // C.CHUNK - -(-p // C.CHUNK) >= 2
            assert c.expect()[0] == (0 if tail == "copy" else S.E_DATA_MALFORMED)
    entered = [c for c in cases if c.name.startswith("chunk entered at offset 4095")]
    assert [c.expect()[0] for c in entered] == [0, S.E_DATA_MALFORMED, S.E_OUTPUT_OVERRUN]
    for c in entered:  # the first tag starting in chunk 2 is a copy-1 at its last byte
        first = min(st for st, *_ in c.s.tags if st >= 2 * C.CHUNK)
        assert first == 3 * C.CHUNK - 1 and c.s.tags[[t[0] for t in c.s.tags].index(first)][2] == 1
    full = [c for c in cases if c.name.startswith("2048 copy-1 tags")]
    seen = set()
    for c in full:
        in_chunk = [i for i, t in enumerate(c.s.tags) if 2 * C.CHUNK <= t[0] < 3 * C.CHUNK]
        assert len(in_chunk) == 2048 and all(c.s.tags[i][2] == 1 for i in in_chunk)
        rc, i, _ = c.expect()
        seen.add((rc, None if i is None else i - in_chunk[0]))
    assert seen == {(0, None)} | {(rc, t) for rc in (S.E_DATA_MALFORMED, S.E_OUTPUT_OVERRUN) for t in (0, 63, 64, 65, 2047)}
    two = {c.name: c for c in cases if c.name.startswith("failures in chunks")}
    for name, rc in (("-3 then -5", S.E_OUTPUT_OVERRUN), ("-5 then -3", S.E_DATA_MALFORMED)):
        c = two[f"failures in chunks 1 and 3, {name}"]
        _, i, _ = c.expect()
        assert c.expect()[0] == rc and c.s.tags[i][0] // C.CHUNK == 1
        # the other failure is a copy-4 in chunk 3 that fails on its own: a bad offset, or no space
        (j, (st, _, _, n, off, _)), = [(j, t) for j, t in enumerate(c.s.tags) if t[0] >= 3 * C.CHUNK and t[2] == 4]
        before = sum(t[3] for t in c.s.tags[:j])
        assert st // C.CHUNK == 3 and (off > before if rc == S.E_OUTPUT_OVERRUN else before + n > c.cap)
    cut = [c for c in cases if "terminal header cut" in c.name]
    assert [c.expect()[0] for c in cut] == [S.E_DATA_MALFORMED, S.E_OUTPUT_OVERRUN]
    for c in cut:
        assert c.s.tags[c.expect()[1]][0] < C.CHUNK and len(c.data) - c.s.tags[-1][0] == 3
    lens = {len(c.data) for c in cases if "input bytes" in c.name}
    assert lens == {k * C.CHUNK + d for k in (1, 2, 5) for d in (-1, 0, 1)}
    across = [c for c in cases if "last literal across" in c.name]
    assert len(across) == 2 * 7 and {c.expect()[0] for c in across} == {0, S.E_OUTPUT_OVERRUN}


def test_port_decodes_shifted_and_chunk_cases():
    port = oracle.port()
    pairs = plan()["invalid"][::20] + plan()["edges"][::10] + plan()["copy_matrix"][::50]
    cases = [C.shifted(c, k) for c, k in pairs] + C.chunk_cases(301)
    for c in cases:
        rc, _, out = c.expect()
        got_rc, got = port.decompress_noheader(c.data, c.cap)
        assert got_rc == rc, (c.name, got_rc, rc)
        if rc == 0:
            assert got == out, c.name


def test_big_literal_cases():
    """The table of results for literals of 2^31 bytes or more: -5 once the room holds the length, by construction
    and by the port (whose output buffer of up to 4 GiB is allocated lazily and never touched)."""
    want = {(1 << 31) - 1: (-3, -5, -5), 0xFFFFFFFE: (-3, -3, -3), (1 << 31) + 12345: (-3, -5, -5)}
    port = oracle.port()
    cases = C.big_literal_cases(7)
    assert len(cases) == 9
    for j, c in enumerate(cases):
        field = C.BIG_FIELDS[j // 3]
        rc, i, _ = c.expect()
        assert rc == want[field][j % 3] and i == len(c.s.tags) - 1, c.name
        assert port.decompress_noheader(c.data, c.cap)[0] == rc, c.name


def test_numpy_built_streams():
    r = C.RunStream(1, 1 << 20, n_copies=8)
    rc, got = oracle.port().decompress_noheader(r.data, r.produced)
    assert rc == 0 and len(got) == r.produced
    assert got[:C.CHUNK] == r.head and got[C.CHUNK:r.run_end] == r.head[-1:] * (r.run_end - C.CHUNK)
    for o, x, n in r.copies:
        assert got[o:o + n] == r.head[x:x + n]
    assert got[r.produced - len(r.tail):] == r.tail
    assert oracle.port().decompress_noheader(r.data, r.produced - 1)[0] == S.E_OUTPUT_OVERRUN
    assert oracle.port().decompress_noheader(r.data + r.bad_offset_tail(), r.produced + 8)[0] == S.E_DATA_MALFORMED
    data, cap = C.saturating_stream(2)
    assert (len(data) - 4096 - 18) // 3 * 64 > 1 << 32
    assert oracle.port().decompress_noheader(data, cap)[0] == S.E_OUTPUT_OVERRUN
