"""Seeded input generators shared by the oracle tests, the GPU tests and tests/golden/make_golden.py.

synth_cases() must stay identical to tests/golden/make_golden.py::synth_cases
(golden.json records the reference's output for every entry); reference_cases.json records the
reference's results on the inputs generated below, so changing a generator means regenerating it."""
import functools
import json
import os
import sys

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN_DIR)
from make_golden import synth_cases  # noqa: E402,F401

EDGE_FRAGMENT_SIZES = list(range(0, 40)) + [59, 60, 61, 62, 255, 256, 257, 258] + list(range(4081, 4112)) + \
    list(range(32753, 32769))
EDGE_COMPRESS_SIZES = (0, 1, 32767, 32768, 32769, 65536, 70001, 150000)


@functools.lru_cache(maxsize=None)
def reference_cases() -> dict:
    """tests/golden/reference_cases.json: the reference's results on the generated inputs of this module."""
    with open(os.path.join(GOLDEN_DIR, "reference_cases.json")) as f:
        return json.load(f)


def edge_text() -> bytes:
    rng = np.random.default_rng(7)
    return bytes(rng.integers(97, 101, 40000, dtype=np.uint8))


def edge_compress_input(text: bytes, n: int) -> bytes:
    return text[:n] * (n // 40000 + 1)


def corrupted_fragments(compress_fragment):
    """(stream, capacity) pairs: wm-13 fragments of 1500-byte fuzz pages with a byte replaced, the tail cut or two
    bytes replaced, decoded into the page size, half of it or a little more."""
    rng = np.random.default_rng(99)
    out = []
    for page in fuzz_pages(5, 14, 1500):
        c = bytearray(compress_fragment(page, 13))
        for _ in range(60):
            d = bytearray(c)
            mode = int(rng.integers(0, 3))
            if mode == 0 and len(d):
                d[int(rng.integers(0, len(d)))] = int(rng.integers(0, 256))
            elif mode == 1 and len(d) > 1:
                d = d[: int(rng.integers(1, len(d)))]
            elif len(d) > 4:
                i = int(rng.integers(0, len(d) - 2))
                d[i:i + 2] = bytes(rng.integers(0, 256, 2, dtype=np.uint8))
            cap = int(rng.choice([len(page), len(page) // 2, len(page) + 100]))
            out.append((bytes(d), cap))
    return out


def ends_inside_tag(s: bytes) -> bool:
    """True when walking tags from the start runs off the end inside a tag's trailing bytes."""
    pos, n = 0, len(s)
    while pos < n:
        t = s[pos]
        pos += 1
        k = t & 3
        if k == 0:
            ln = (t >> 2) + 1
            if ln > 60:
                nb = ln - 60
                if pos + nb > n:
                    return True
                ln = int.from_bytes(s[pos:pos + nb], "little") + 1
                pos += nb
            if pos + ln > n:
                return False  # literal payload cut: defined (-5) in the reference
            pos += ln
        else:
            nb = (1, 2, 4)[k - 1]
            if pos + nb > n:
                return True
            pos += nb
    return False


def ends_inside_tag_header(s: bytes) -> bool:
    """True when the end of input cuts a tag's header (tag byte + offset / length bytes): the reference's
    UB case (csnappy_decompress.c:331-342,350).  Payload shortage of a literal is NOT that case (-5, :374)."""
    pos, n = 0, len(s)
    while pos < n:
        tag = s[pos]
        kind = tag & 3
        if kind == 0:
            ln = (tag >> 2) + 1
            hdr = 1
            if ln > 60:
                nb = ln - 60
                if pos + 1 + nb > n:
                    return True
                ln = int.from_bytes(s[pos + 1: pos + 1 + nb], "little") + 1
                hdr = 1 + nb
            pos += hdr + (ln & 0xFFFFFFFF)
        else:
            hdr = (2, 3, 5)[kind - 1]
            if pos + hdr > n:
                return True
            pos += hdr
    return False


def corrupt_streams(compress_fragment, size, wm, seed, count):
    """Fragments of fuzz pages, in turn: valid, a byte flipped, the tail cut, valid with an under-sized capacity,
    three bytes replaced, random bytes appended.  -> (streams, capacities)"""
    pages = fuzz_pages(seed, count, size)
    comp = [compress_fragment(p, wm) for p in pages]
    rng = np.random.default_rng(seed + 1)
    streams, caps = [], []
    for i, c in enumerate(comp):
        d = bytearray(c)
        k = i % 6
        if k == 1 and len(d) > 8:
            d[int(rng.integers(0, len(d)))] ^= int(rng.integers(1, 256))
        elif k == 2 and len(d) > 8:
            d = d[: int(rng.integers(1, len(d)))]
        elif k == 4 and len(d) > 8:
            for _ in range(3):
                d[int(rng.integers(0, len(d)))] = int(rng.integers(0, 256))
        elif k == 5:
            d += bytes(rng.integers(0, 256, int(rng.integers(1, 9)), dtype=np.uint8))
        streams.append(bytes(d))
        caps.append(size if k != 3 else int(rng.integers(1, size)))
    return streams, caps


# (size, wm) -> (seed, count) of corrupt_streams() in tests/test_gpu_canaries.py::test_decode_never_writes_at_or_past_cap
CANARY_DECODE = {(4096, 13): (515 + 4096, 84), (32768, 15): (515 + 32768, 28)}


def fuzz_pages(seed: int, count: int, size: int):
    """Mixed-entropy pages: random, zero, periodic, low-entropy, word text, copies-with-noise."""
    rng = np.random.default_rng(seed)
    words = [bytes(rng.integers(97, 123, int(rng.integers(2, 10)), dtype=np.uint8)) for _ in range(300)]
    out = []
    for i in range(count):
        k = i % 7
        if k == 0:
            b = rng.integers(0, 256, size, dtype=np.uint8).tobytes()
        elif k == 1:
            b = bytes(size)
        elif k == 2:
            p = int(rng.integers(1, 80))
            pat = rng.integers(0, 256, p, dtype=np.uint8).tobytes()
            b = (pat * (size // p + 1))[:size]
        elif k == 3:
            b = rng.integers(0, int(rng.integers(2, 6)), size, dtype=np.uint8).tobytes()
        elif k == 4:
            b = b" ".join(words[int(j)] for j in rng.integers(0, 300, size // 2 + 8))[:size]
        elif k == 5:
            base = bytearray(b" ".join(words[int(j)] for j in rng.integers(0, 40, size // 2 + 8))[:size])
            for j in rng.integers(0, max(size, 1), size // 50):
                base[int(j)] = int(rng.integers(0, 256))
            b = bytes(base)
        else:
            # long matches at long offsets + runs
            half = rng.integers(0, 256, max(size // 3, 1), dtype=np.uint8).tobytes()
            b = (half + bytes(int(rng.integers(0, 200))) + half + half[::-1] + half)[:size]
            b = b + bytes(size - len(b))
        out.append(b)
    return out
