"""Restatement and staging helpers for the batched framing calls (csnappy_framed_batch_*): the declared-length walk, and
the layouts a batch test needs (odd input offsets, output slots with gaps).  Plain Python and numpy; no torch."""
from __future__ import annotations

import numpy as np

import framed as F


def declared_length(s: bytes) -> tuple[int, int]:
    """csnappy_framed_batch_decompressed_length restated: the chunk walk of read_framed with unbounded capacity and no
    decoding.  -> (sum of the data lengths the headers declare up to the first walk failure, 0 or -5)."""
    s = bytes(s)
    pos = total = 0
    while pos < len(s):
        if len(s) - pos < 4:
            return total, F.E_DATA_MALFORMED
        t = s[pos]
        blen = int.from_bytes(s[pos + 1:pos + 4], "little")
        body = s[pos + 4:pos + 4 + blen]
        if len(body) < blen or (pos == 0 and t != 0xFF):
            return total, F.E_DATA_MALFORMED
        if t == 0xFF:
            if body != b"sNaPpY":
                return total, F.E_DATA_MALFORMED
        elif t <= 1:
            if blen < (5 if t == 0 else 4):
                return total, F.E_DATA_MALFORMED
            if t == 0:
                v = F.parse_varint(body[4:])
                if v is None or v[0] > F.CHUNK:
                    return total, F.E_DATA_MALFORMED
                total += v[0]
            else:
                if blen - 4 > F.CHUNK:
                    return total, F.E_DATA_MALFORMED
                total += blen - 4
        elif t <= 0x7F:
            return total, F.E_DATA_MALFORMED
        pos += 4 + blen
    return total, 0


def packed(bufs, seed: int, pad: int = 7) -> tuple[bytes, list[int]]:
    """The buffers behind each other with 1..pad random bytes in front of each one (odd offsets included)."""
    rng = np.random.default_rng(seed)
    parts, offs, at = [], [], 0
    for b in bufs:
        g = int(rng.integers(1, pad + 1))
        parts.append(rng.integers(0, 256, g, dtype=np.uint8).tobytes())
        at += g
        offs.append(at)
        parts.append(bytes(b))
        at += len(b)
    return b"".join(parts) + b"\0" * 8, offs


def slots_with_gaps(sizes, seed: int, gap: int = 19) -> tuple[list[int], int]:
    """Output offsets for slots of the given sizes with 0..gap bytes between them; -> (offsets, end of the last)."""
    rng = np.random.default_rng(seed)
    offs, at = [], int(rng.integers(0, gap + 1))
    for n in sizes:
        offs.append(at)
        at += int(n) + int(rng.integers(0, gap + 1))
    return offs, at


def untouched_outside(raw: bytes, spans, fill: int = 0xA5) -> list[int]:
    """Indices of bytes outside every [start, end) span that no longer hold `fill` (first few)."""
    a = np.frombuffer(raw, dtype=np.uint8)
    keep = np.ones(len(a), dtype=bool)
    for s, e in spans:
        keep[s:e] = False
    bad = np.nonzero(keep & (a != fill))[0]
    return bad[:10].tolist()
