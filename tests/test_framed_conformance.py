"""CPU checks of the framing-format restatement (tests/framed.py): CRC-32C and its mask against the standard
vectors, the writer against csnappy_compress and the 1/8 type rule, the reader on every hostile class."""
from __future__ import annotations

import numpy as np
import pytest

import framed as F
import oracle
import streams

CRC_VECTORS = [
    (b"123456789", 0xE3069283),
    (bytes(32), 0x8A9136AA),
    (b"\xff" * 32, 0x62A8AB43),
    (bytes(range(32)), 0x46DD794E),
    (bytes(range(31, -1, -1)), 0x113FDB5C),
    (b"", 0),
    (b"a", 0xC1D04330),
]


@pytest.mark.parametrize("data,crc", CRC_VECTORS)
def test_crc32c_vectors(data, crc):
    assert F.crc32c(data) == crc == F.crc32c_scalar(data)


def test_mask_vectors():
    assert F.mask(0) == 0xA282EAD8
    assert F.mask(0xC1D04330) == 0x28E46E78


def test_crc32c_many_matches_scalar():
    rng = np.random.default_rng(5)
    bufs = [rng.integers(0, 256, int(n), dtype=np.uint8).tobytes() for n in list(range(0, 40)) + [999, 4096, 5000]]
    assert F.crc32c_many(bufs) == [F.crc32c_scalar(b) for b in bufs]


def _parse(s: bytes):
    assert s[:10] == F.IDENT
    out, pos = [], 10
    while pos < len(s):
        t, n = s[pos], int.from_bytes(s[pos + 1:pos + 4], "little")
        out.append((t, s[pos + 4:pos + 8], s[pos + 8:pos + 4 + n]))
        pos += 4 + n
    return out


@pytest.mark.parametrize("wm", [9, 12, 16])
def test_writer_against_csnappy_compress(wm):
    port = oracle.port()
    for n in F.LENGTHS:
        data = F.mixed_bytes(n + wm, n, scale=20000)
        s = F.write_framed(data, wm, port)
        assert len(s) <= F.max_length(n)
        recs = _parse(s)
        assert len(recs) == -(-n // F.CHUNK)
        for k, (t, crc, payload) in enumerate(recs):
            chunk = data[k * F.CHUNK:(k + 1) * F.CHUNK]
            z = port.compress(chunk, wm)
            m = len(chunk)
            assert t == (0 if len(z) < m - m // 8 else 1)
            assert payload == (z if t == 0 else chunk)
            assert int.from_bytes(crc, "little") == F.mask(F.crc32c(chunk))
        r = F.read_framed(s, n)
        assert r.key() == (0, n, None) and r.data == data


def test_max_length_is_reached_by_incompressible_input():
    data = np.random.default_rng(1).integers(0, 256, 2 * F.CHUNK + 5, dtype=np.uint8).tobytes()
    assert len(F.write_framed(data, 16)) == F.max_length(len(data))


@pytest.mark.parametrize("n", [F.CHUNK, 4096])
def test_edge_chunks_sit_on_the_type_rule(n):
    port = oracle.port()
    for d in (-1, 0, 1):
        c = F.edge_chunk(n, 16, d, port=port)
        assert c is not None, (n, d)
        assert len(port.compress(c, 16)) == n - n // 8 + d
        assert F.write_framed(c, 16, port)[10] == (0 if d < 0 else 1)


def test_every_hostile_class_occurs():
    hs = F.hostile_streams(3, 16, stream_cases=streams.boundary_streams(3)[:12])
    assert {h.cls for h in hs} >= F.HOSTILE_CLASSES


def test_reader_on_hostile_streams():
    hs = {h.cls: h for h in F.hostile_streams(4, 16, stream_cases=streams.boundary_streams(4)[:8])}
    valid = F.read_framed(hs["valid"].stream, hs["valid"].cap)
    assert valid.rc == 0 and valid.out_length == hs["valid"].cap
    assert F.read_framed(hs["empty"].stream, 0).key() == (0, 0, None)
    assert F.read_framed(hs["no_identifier"].stream, hs["valid"].cap).key() == (F.E_DATA_MALFORMED, 0, 0)
    assert F.read_framed(hs["capacity_short"].stream, hs["capacity_short"].cap).rc == F.E_OUTPUT_INSUF
    for cls in ("repeated_identifier", "concatenated", "foreign_chunking", "skippable_fe_16777215", "stored_65536"):
        assert F.read_framed(hs[cls].stream, hs[cls].cap).rc == 0, cls
    for cls in ("reserved_02", "reserved_7f", "bad_identifier_body_mid", "stored_65537", "varint_65537", "varint_short",
                "varint_long", "bad_varint_cut"):
        assert F.read_framed(hs[cls].stream, hs[cls].cap).rc == F.E_DATA_MALFORMED, cls
    a = F.read_framed(hs["two_failures_crc_decode"].stream, hs["valid"].cap)
    b = F.read_framed(hs["two_failures_decode_crc"].stream, hs["valid"].cap)
    assert a.rc == F.E_CHECKSUM and b.rc == F.E_DATA_MALFORMED and a.failed_offset == b.failed_offset > 10
    assert a.out_length == b.out_length > 0
