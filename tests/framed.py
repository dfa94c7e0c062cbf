"""Plain restatements of the Snappy framing format as include/csnappy_batch.h pins it, and seeded generators of the
streams where a framed writer or reader goes wrong.  Plain Python and numpy on top of the oracle port; no torch.

* ``crc32c`` / ``mask``  CRC-32C (Castagnoli, reflected 0x82F63B78, init ~0, final ~0) and the format's mask;
  ``crc32c_many`` runs slicing-by-8 over many buffers at once with numpy.
* ``write_framed``       the writer: identifier, then per 64 KiB chunk csnappy_compress (the port) when it is shorter
  than n - n/8, else the chunk itself, each behind its masked CRC.
* ``read_framed``        the reader: the chunk walk with every framing rule, then per data chunk decode (the port),
  length and CRC checks; the failing chunk with the smallest header position wins.
* generators             lengths, chunks at the edge of the type rule, foreign-style chunking and hostile streams.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass

import numpy as np

import oracle
from containers import mixed_bytes, varint32

CHUNK = 65536
IDENT = b"\xff\x06\x00\x00sNaPpY"
E_OUTPUT_INSUF, E_DATA_MALFORMED, E_CHECKSUM = -2, -5, -102
POLY = 0x82F63B78


# ------------------------------------------------------------------------------------------------------- CRC-32C
def _tables() -> np.ndarray:
    t = np.zeros((8, 256), dtype=np.uint32)
    for i in range(256):
        r = i
        for _ in range(8):
            r = (r >> 1) ^ POLY if r & 1 else r >> 1
        t[0, i] = r
    for k in range(1, 8):
        t[k] = (t[k - 1] >> 8) ^ t[0][t[k - 1] & 0xFF]
    return t


T = _tables()


def crc32c_scalar(data: bytes) -> int:
    r = 0xFFFFFFFF
    for b in data:
        r = int(T[0][(r ^ b) & 0xFF]) ^ (r >> 8)
    return r ^ 0xFFFFFFFF


def crc32c_many(bufs) -> list[int]:
    """CRC-32C of every buffer.  Buffers of 4 bytes or more run together: the ~0 init equals complementing the first
    four bytes from register 0, and zero bytes in front of a buffer leave register 0 alone, so every buffer is
    right-aligned in one matrix and slicing-by-8 runs over its 8-byte columns."""
    bufs = [bytes(b) for b in bufs]
    out = [0] * len(bufs)
    big = [i for i, b in enumerate(bufs) if len(b) >= 4]
    for i, b in enumerate(bufs):
        if len(b) < 4:
            out[i] = crc32c_scalar(b)
    if not big:
        return out
    width = (max(len(bufs[i]) for i in big) + 7) // 8 * 8
    m = np.zeros((len(big), width), dtype=np.uint8)
    for row, i in enumerate(big):
        b = np.frombuffer(bufs[i], dtype=np.uint8).copy()
        b[:4] ^= 0xFF
        m[row, width - len(b):] = b
    w = m.view("<u4")
    r = np.zeros(len(big), dtype=np.uint32)
    for j in range(0, width // 4, 2):
        a = w[:, j] ^ r
        b = w[:, j + 1]
        r = (T[7][a & 0xFF] ^ T[6][(a >> 8) & 0xFF] ^ T[5][(a >> 16) & 0xFF] ^ T[4][a >> 24] ^
             T[3][b & 0xFF] ^ T[2][(b >> 8) & 0xFF] ^ T[1][(b >> 16) & 0xFF] ^ T[0][b >> 24])
    for row, i in enumerate(big):
        out[i] = int(r[row]) ^ 0xFFFFFFFF
    return out


def crc32c(data: bytes) -> int:
    return crc32c_many([data])[0]


def mask(crc: int) -> int:
    return ((((crc >> 15) | (crc << 17)) & 0xFFFFFFFF) + 0xA282EAD8) & 0xFFFFFFFF


def max_length(n: int) -> int:
    return 10 + 8 * (-(-n // CHUNK)) + n


# ------------------------------------------------------------------------------------------------- writer / reader
def chunk_record(kind: int, crc: int, payload: bytes) -> bytes:
    body = struct.pack("<I", crc) + payload
    return bytes([kind]) + len(body).to_bytes(3, "little") + body


def write_framed(data: bytes, wm: int, port=None) -> bytes:
    port = port or oracle.port()
    chunks = [data[at:at + CHUNK] for at in range(0, len(data), CHUNK)]
    crcs = crc32c_many(chunks)
    out = [IDENT]
    for c, crc in zip(chunks, crcs):
        z = port.compress(c, wm)
        n = len(c)
        out.append(chunk_record(0, mask(crc), z) if len(z) < n - n // 8 else chunk_record(1, mask(crc), c))
    return b"".join(out)


def parse_varint(p: bytes):
    """csnappy_get_uncompressed_length: -> (value, bytes used) or None."""
    v = shift = used = 0
    while True:
        if shift >= 32 or used == len(p):
            return None
        c = p[used]
        used += 1
        v = (v | ((c & 0x7F) << shift)) & 0xFFFFFFFF
        if c < 128:
            return v, used
        shift += 7


@dataclass
class ReadResult:
    rc: int
    out_length: int
    failed_offset: int | None
    data: bytes = b""  # the valid prefix, dst[0, out_length)

    def key(self):
        return self.rc, self.out_length, self.failed_offset


def read_framed(s: bytes, cap: int, decode=None) -> ReadResult:
    decode = decode or oracle.port().decompress_noheader
    s = bytes(s)
    pos = produced = 0
    fails, chunks = [], []  # (position, rc); (position, kind, payload, out length, stored crc, output offset)
    while pos < len(s):
        if len(s) - pos < 4:
            fails.append((pos, E_DATA_MALFORMED))
            break
        t = s[pos]
        blen = int.from_bytes(s[pos + 1:pos + 4], "little")
        body = s[pos + 4:pos + 4 + blen]
        if len(body) < blen or (pos == 0 and t != 0xFF):
            fails.append((pos, E_DATA_MALFORMED))
            break
        if t == 0xFF:
            if body != b"sNaPpY":
                fails.append((pos, E_DATA_MALFORMED))
                break
        elif t <= 1:
            if blen < (5 if t == 0 else 4):
                fails.append((pos, E_DATA_MALFORMED))
                break
            crc, payload = struct.unpack_from("<I", body)[0], body[4:]
            if t == 0:
                v = parse_varint(payload)
                if v is None or v[0] > CHUNK:
                    fails.append((pos, E_DATA_MALFORMED))
                    break
                olen = v[0]
                payload = payload[v[1]:]
            else:
                if len(payload) > CHUNK:
                    fails.append((pos, E_DATA_MALFORMED))
                    break
                olen = len(payload)
            if olen > cap - produced:
                fails.append((pos, E_OUTPUT_INSUF))
                break
            chunks.append((pos, t, payload, olen, crc, produced))
            produced += olen
        elif t <= 0x7F:
            fails.append((pos, E_DATA_MALFORMED))
            break
        pos += 4 + blen
    outs = {}
    for at, t, payload, olen, crc, _ in chunks:
        if t == 0:
            rc, out = decode(payload, olen)
            if rc != 0 or len(out) != olen:
                fails.append((at, E_DATA_MALFORMED))
                continue
            outs[at] = out
        else:
            outs[at] = payload
    good = [c for c in chunks if c[0] in outs]
    for c, crc in zip(good, crc32c_many([outs[c[0]] for c in good])):
        if mask(crc) != c[4]:
            fails.append((c[0], E_CHECKSUM))
    if not fails:
        return ReadResult(0, produced, None, b"".join(outs[c[0]] for c in chunks))
    at, rc = min(fails)
    before = [c for c in chunks if c[0] < at]
    return ReadResult(rc, sum(c[3] for c in before), at, b"".join(outs[c[0]] for c in before))


# ------------------------------------------------------------------------------------------------------- generators
LENGTHS = (0, 1, 7, 8, 9, 32767, 32768, 32769, 65535, 65536, 65537, 131072, 3 * 2**20 + 4097)


def edge_chunk(n: int, wm: int, d: int, seed: int = 0, port=None) -> bytes | None:
    """A chunk of n bytes whose csnappy_compress size is n - n//8 + d: random bytes with a run of one byte value
    planted inside; each byte of run saves about one byte, so the run length is bisected, then scanned."""
    port = port or oracle.port()
    target = n - n // 8 + d
    for s in range(16):
        rng = np.random.default_rng([seed, n, wm, s])
        base = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        at = int(rng.integers(0, 64))
        v = bytes([int(rng.integers(0, 256))])

        def size(r):
            return len(port.compress(base[:at] + v * r + base[at + r:], wm))

        lo, hi = 0, n - at
        while hi - lo > 1:  # size is about decreasing in the run length
            mid = (lo + hi) // 2
            if size(mid) > target:
                lo = mid
            else:
                hi = mid
        for r in range(max(0, lo - 64), min(n - at, lo + 64)):
            if size(r) == target:
                return base[:at] + v * r + base[at + r:]
    return None


def foreign_framed(seed: int, data: bytes, port=None) -> bytes:
    """Valid stream as another writer might chunk it: ragged chunk sizes 1..65536 (both ends included), a random
    choice of compressed / stored per chunk, padding and a repeated identifier between chunks."""
    port = port or oracle.port()
    rng = np.random.default_rng(seed)
    sizes, at = [], 0
    while at < len(data):
        n = int(rng.choice([1, 2, CHUNK, int(rng.integers(1, CHUNK + 1)), int(rng.integers(1, 300))]))
        sizes.append(min(n, len(data) - at))
        at += sizes[-1]
    chunks = []
    at = 0
    for n in sizes:
        chunks.append(data[at:at + n])
        at += n
    crcs = crc32c_many(chunks)
    out = [IDENT]
    for c, crc in zip(chunks, crcs):
        if rng.random() < 0.5:
            out.append(chunk_record(0, mask(crc), port.compress(c, int(rng.integers(9, 17)))))
        else:
            out.append(chunk_record(1, mask(crc), c))
        r = rng.random()
        if r < 0.1:
            out.append(bytes([0xFE]) + (3).to_bytes(3, "little") + b"\0\0\0")
        elif r < 0.15:
            out.append(IDENT)
    return b"".join(out)


def _chunks(s: bytes):
    """[(position, type, body length)] of a well-formed stream."""
    out, pos = [], 0
    while pos < len(s):
        blen = int.from_bytes(s[pos + 1:pos + 4], "little")
        out.append((pos, s[pos], blen))
        pos += 4 + blen
    return out


@dataclass
class Hostile:
    cls: str
    stream: bytes
    cap: int


def _data_record(body_payload: bytes, kind: int, out: bytes, crc_ok: bool = True) -> bytes:
    c = mask(crc32c(out))
    return chunk_record(kind, c if crc_ok else c ^ 1, body_payload)


def skip_chunk(t: int, n: int, fill: int = 0x5A) -> bytes:
    return bytes([t]) + n.to_bytes(3, "little") + bytes([fill]) * n


def hostile_streams(seed: int, wm: int = 16, port=None, stream_cases=None) -> list[Hostile]:
    """Every class of hostile stream the reader must handle.  The base is a written stream of 5 chunks (compressed
    and stored ones); `stream_cases` (tests/streams.py Cases) become compressed chunks with every tag form."""
    port = port or oracle.port()
    rng = np.random.default_rng(seed)
    data = mixed_bytes(seed, 3 * CHUNK + 777, scale=CHUNK // 2) + rng.integers(0, 256, CHUNK, dtype=np.uint8).tobytes()
    base = write_framed(data, wm, port)
    ch = _chunks(base)
    total = len(data)
    out = []

    def add(cls, s, cap=None):
        out.append(Hostile(cls, bytes(s), total if cap is None else cap))

    add("valid", base)
    add("no_identifier", base[10:])
    add("bad_identifier_body_start", base[:4] + b"sNaPpZ" + base[10:])
    add("bad_identifier_length_start", b"\xff\x07\x00\x00sNaPpYY" + base[10:])
    mid = ch[2][0]
    add("bad_identifier_body_mid", base[:mid] + b"\xff\x06\x00\x00snappy" + base[mid:])
    add("bad_identifier_length_mid", base[:mid] + b"\xff\x05\x00\x00sNaPp" + base[mid:])
    add("repeated_identifier", base[:mid] + IDENT + base[mid:])
    add("concatenated", base + base, 2 * total)
    for t in (0xFE, 0x80, 0xFD):
        for n in (0, 1, 65536, (1 << 24) - 1):
            add(f"skippable_{t:02x}_{n}", base[:mid] + skip_chunk(t, n) + base[mid:])
    for t in (0x02, 0x7F):
        add(f"reserved_{t:02x}", base[:mid] + skip_chunk(t, 4) + base[mid:])
    for t in (0, 1):
        for n in range(5):
            add(f"body_{t}_{n}", base[:mid] + bytes([t]) + n.to_bytes(3, "little") + bytes(n) + base[mid:])
    big = rng.integers(0, 256, CHUNK + 1, dtype=np.uint8).tobytes()
    add("stored_65537", base[:mid] + _data_record(big, 1, big) + base[mid:], total + CHUNK + 1)
    full = rng.integers(0, 256, CHUNK, dtype=np.uint8).tobytes()
    add("stored_65536", base[:mid] + _data_record(full, 1, full) + base[mid:], total + CHUNK)
    small = b"abcdefgh" * 16
    z = port.compress(small, wm)[len(varint32(len(small))):]  # the raw stream, without its varint
    add("bad_varint_long", base[:mid] + _data_record(b"\x80\x80\x80\x80\x80\x01" + z, 0, small) + base[mid:])
    add("bad_varint_cut", base[:mid] + _data_record(b"\x80\x80", 0, small) + base[mid:])
    v65537 = varint32(CHUNK + 1) + port.compress(big, wm)[3:]
    add("varint_65537", base[:mid] + _data_record(v65537, 0, big) + base[mid:], total + CHUNK + 1)
    for d in (-1, 1):
        add(f"varint_{'short' if d < 0 else 'long'}", base[:mid] + _data_record(varint32(len(small) + d) + z, 0, small)
            + base[mid:], total + len(small) + 1)
    for i, c in enumerate(stream_cases or []):
        rc, _, produced = c.expect(0xFFFF)
        if rc != 0 or not produced or len(produced) > CHUNK:
            continue
        rec = _data_record(varint32(len(produced)) + c.data, 0, produced)
        add("tag_forms", IDENT + rec, len(produced))
        if i % 4 == 0:
            for d in (-1, 1):
                add("tag_forms_varint_off", IDENT + _data_record(varint32(len(produced) + d) + c.data, 0, produced),
                    len(produced) + 1)
    for pos, _, _ in ch:
        for k in range(4):
            add("truncated_header", base[:pos + k])
        add("truncated_body", base[:pos + 4 + 2])
    for i, (pos, t, _) in enumerate(ch[1:], 1):
        s = bytearray(base)
        s[pos + 4 + int(rng.integers(0, 4))] ^= 1 << int(rng.integers(0, 8))
        add(f"crc_bit_{t}", s)
        s = bytearray(base)
        s[pos + 8 + int(rng.integers(4, 200))] ^= 1 << int(rng.integers(0, 8))
        add(f"data_bit_{t}", s)
    add("capacity_short", base, total - 1)
    add("capacity_exact", base, total)
    add("capacity_zero", base, 0)
    c1, c2 = ch[2][0], ch[4][0]
    bad = _data_record(varint32(64) + bytes([0xFE, 0xFF, 0xFF]), 0, bytes(64))  # copy before any output: -5

    def crc_flipped(at):
        n = 4 + int.from_bytes(base[at + 1:at + 4], "little")
        r = bytearray(base[at:at + n])
        r[4] ^= 0x10
        return bytes(r), n

    for first, second in (("crc", "decode"), ("decode", "crc")):
        parts, at = [], 0
        for what, pos in ((first, c1), (second, c2)):
            rec, n = crc_flipped(pos)
            parts += [base[at:pos], rec if what == "crc" else bad]
            at = pos + n
        add(f"two_failures_{first}_{second}", b"".join(parts) + base[at:])
    s = bytearray(base)
    s[c1 + 4] ^= 0x10
    add("two_failures_crc_reserved", bytes(s[:c2]) + skip_chunk(0x03, 2) + bytes(s[c2:]))
    s = bytearray(base)
    s[c2 + 4] ^= 0x10
    add("two_failures_reserved_crc", bytes(s[:c1]) + skip_chunk(0x03, 2) + bytes(s[c1:]))
    add("foreign_chunking", foreign_framed(seed, data[:2 * CHUNK + 999], port), 2 * CHUNK + 999)
    add("empty", b"", 0)
    add("identifier_only", IDENT, 0)
    return out


HOSTILE_CLASSES = {
    "valid", "no_identifier", "bad_identifier_body_start", "bad_identifier_length_start", "bad_identifier_body_mid",
    "bad_identifier_length_mid", "repeated_identifier", "concatenated", "reserved_02", "reserved_7f", "stored_65537",
    "stored_65536", "bad_varint_long", "bad_varint_cut", "varint_65537", "varint_short", "varint_long", "tag_forms",
    "tag_forms_varint_off", "truncated_header", "truncated_body", "capacity_short", "capacity_exact",
    "two_failures_crc_reserved", "two_failures_reserved_crc", "two_failures_crc_decode",
    "two_failures_decode_crc", "foreign_chunking", "empty", "identifier_only",
} | {f"skippable_{t:02x}_{n}" for t in (0xFE, 0x80, 0xFD) for n in (0, 1, 65536, (1 << 24) - 1)} | {
    f"body_{t}_{n}" for t in (0, 1) for n in range(5)} | {"crc_bit_0", "crc_bit_1", "data_bit_0", "data_bit_1"}
