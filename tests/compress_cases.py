"""Compressor inputs built by construction, and a plain Python restatement of csnappy_compress_fragment.

compress_fragment() follows csnappy_compress.c:469-606 (and oracle/snappy_oracle.c) statement by statement and can
record a trace of every table touch, copy and literal.  The generators below plant structures into incompressible
random filler at probe positions computed from the reference's skip schedule, so that the greedy parse is forced
through the compressor kernel's rarely taken paths:

* several probes on one hash slot inside one window of 32 probes (pairs at every distance, three and four colliding
  words, a true repeat plus a collision, A-B-A / A-A-B / B-A-A orders, interleaved and nested pairs), at the block
  start, right behind a copy (the insert of ip-1 and the re-probe of ip), after a short in-window copy, and in
  strided windows (skip stride 2, 3, 4);
* short copies inside a window, chains of re-probe hits, and a copy that skips a position sharing a slot with a
  later probe;
* the scan end: no hit up to ip_limit, a hit at the last valid probe, copies that end at ip_limit - 1, ip_limit
  and n, a candidate at position 0;
* match lengths at the kernel's extension steps (4 + G, 4 + 5G for G = 8, 16, 32), literal and copy lengths at
  every header and split boundary, offsets at the copy-1 / copy-2 limit, and 31..65 copies per block.

Every episode states what the parse must do (a copy at a given position, or touches at given positions); after
each episode the block is compressed with trace and the episode is redrawn if its plan did not happen.

Literal lengths in front of a copy are not free: a copy starts at a probe position, so the literal is 0 (re-probe
hit) or 1 + the distance of a probe from its scan start: 1..33, odd values to 97, 97 + 3k to 193, 193 + 4k, ...
(reachable_literals()).  60, 128, 129 and 256 never precede a copy; they occur as final literals.
"""
import functools

import numpy as np

MUL = 0x1E35A7BD
MARGIN = 15  # kInputMarginBytes, csnappy_compress.c:468
GS = (8, 16, 32)


def slot(v: int, wm: int) -> int:
    return ((v * MUL) & 0xFFFFFFFF) >> (33 - wm)


def u32(d, p: int) -> int:
    return d[p] | d[p + 1] << 8 | d[p + 2] << 16 | d[p + 3] << 24


def _literal(out, d, src, ln):
    v = ln - 1
    if v < 60:
        out.append(v << 2)
    else:
        nb = (v.bit_length() + 7) // 8
        out.append((59 + nb) << 2)
        out += v.to_bytes(nb, "little")
    out += d[src:src + ln]


def _copy(out, off, ln):
    def piece(m):
        if m < 12 and off < 2048:
            out.extend((1 | (m - 4) << 2 | (off >> 8) << 5, off & 0xFF))
        else:
            out.extend((2 | (m - 1) << 2, off & 0xFF, off >> 8))
    while ln >= 68:
        piece(64)
        ln -= 64
    if ln > 64:
        piece(60)
        ln -= 60
    piece(ln)


def compress_fragment(data: bytes, wm: int, trace=None) -> bytes:
    """csnappy_compress_fragment(data, wm).  trace (a list) receives, in order:
    ("t", pos, slot, idx, cand, hit)  a table touch: idx >= 0 is a scan probe (its index in the skip schedule),
                                      -2 the post-copy insert of ip-1 (cand None), -1 the post-copy re-probe of ip;
    ("c", ip, cand, len, op)          a copy, op = output offset of its first tag;
    ("l", len, op, final)             a literal."""
    d = bytes(data) + bytes(4)
    n = len(data)
    out = bytearray()
    tr = trace.append if trace is not None else (lambda e: None)
    if n < MARGIN:
        if n:
            tr(("l", n, 0, True))
            _literal(out, d, 0, n)
        return bytes(out)
    table = [0] * (1 << (wm - 1))
    ip_limit = n - MARGIN
    ip, next_emit = 1, 0
    while True:
        probes, hit = 32, False
        while True:
            step = probes >> 5
            probes += 1
            if ip + step > ip_limit:
                break
            v = u32(d, ip)
            h = slot(v, wm)
            cand = table[h]
            table[h] = ip
            hit = u32(d, cand) == v
            tr(("t", ip, h, probes - 33, cand, hit))
            if hit:
                break
            ip += step
        if not hit:
            break
        tr(("l", ip - next_emit, len(out), False))
        if ip > next_emit:
            _literal(out, d, next_emit, ip - next_emit)
        while True:
            m = 4
            while ip + m < n and d[cand + m] == d[ip + m]:
                k = min(64, n - ip - m)  # (whole runs at a time: the same result as byte by byte)
                m += k if d[cand + m:cand + m + k] == d[ip + m:ip + m + k] else 1
            tr(("c", ip, cand, m, len(out)))
            _copy(out, ip - cand, m)
            ip += m
            next_emit = ip
            if ip >= ip_limit:
                break
            h = slot(u32(d, ip - 1), wm)
            table[h] = ip - 1
            tr(("t", ip - 1, h, -2, None, False))
            v = u32(d, ip)
            h = slot(v, wm)
            cand = table[h]
            table[h] = ip
            hit = u32(d, cand) == v
            tr(("t", ip, h, -1, cand, hit))
            if not hit:
                break
        if ip >= ip_limit:
            break
        ip += 1
    if next_emit < n:
        tr(("l", n - next_emit, len(out), True))
        _literal(out, d, next_emit, n - next_emit)
    return bytes(out)


def offs(j: int) -> int:
    """Distance of probe index j from its scan's start (strides (32 + i) >> 5)."""
    return sum((32 + i) >> 5 for i in range(j))


@functools.lru_cache(maxsize=None)
def reachable_literals(limit: int = 33000) -> frozenset:
    """Literal lengths that can precede a copy: 0 (re-probe hit) and 1 + offs(j)."""
    out, o, j = {0}, 0, 0
    while o < limit:
        out.add(1 + o)
        o += (32 + j) >> 5
        j += 1
    return frozenset(out)


# ---------------------------------------------------------------------------------------- hash collisions
@functools.lru_cache(maxsize=None)
def collisions(wm: int):
    """Groups of distinct 4-byte words sharing one slot at table size wm: list of lists (at least 4 words each)."""
    rng = np.random.default_rng(1000 + wm)
    v = np.unique(rng.integers(0, 1 << 32, 1 << 21, dtype=np.uint64).astype(np.uint32))
    s = ((v.astype(np.uint64) * MUL) & 0xFFFFFFFF) >> (33 - wm)
    order = np.argsort(s, kind="stable")
    v, s = v[order], s[order]
    starts = np.flatnonzero(np.r_[True, s[1:] != s[:-1]])
    ends = np.r_[starts[1:], len(s)]
    groups = [v[a:b][:6].tolist() for a, b in zip(starts, ends) if b - a >= 4]
    rng.shuffle(groups)
    return groups


@functools.lru_cache(maxsize=None)
def overlap_pairs(wm: int, dist: int):
    """Byte strings S of dist + 4 bytes whose words at 0 and at dist differ and share a slot (dist 1..3)."""
    rng = np.random.default_rng(2000 + 16 * wm + dist)
    need = 1 << (wm - 1)
    found = []
    while len(found) < 64:
        b = rng.integers(0, 256, (need * 4, dist + 4), dtype=np.uint64)
        w0 = b[:, 0] | b[:, 1] << 8 | b[:, 2] << 16 | b[:, 3] << 24
        w1 = b[:, dist] | b[:, dist + 1] << 8 | b[:, dist + 2] << 16 | b[:, dist + 3] << 24
        h0, h1 = ((w0 * MUL) & 0xFFFFFFFF) >> (33 - wm), ((w1 * MUL) & 0xFFFFFFFF) >> (33 - wm)
        for r in np.flatnonzero((h0 == h1) & (w0 != w1))[: 64 - len(found)]:
            found.append(bytes(b[r].astype(np.uint8)))
    return found


# ---------------------------------------------------------------------------------------- builder
class Plan(Exception):
    """An episode that cannot be laid out here."""


class Builder:
    """One block under construction: random filler, a parse state known from the skip schedule, and the episodes'
    expectations.  State: e = end of the last copy (None at the block start), s = first scan probe position."""

    def __init__(self, rng, n: int, wm: int):
        self.rng, self.n, self.wm = rng, n, wm
        self.d = bytearray(rng.integers(0, 256, n, dtype=np.uint8).tobytes())
        self.limit = n - MARGIN
        self.e, self.s, self.ne = None, 1, 0
        self.used = set()  # planted positions of the current scan (not usable as a copy source)
        self.groups = iter(collisions(wm))
        self.copies = []  # planned (ip, cand, len)
        self.touch = []   # planned touched positions
        self.runs = set()  # bytes of the offset-1 / -2 runs already used
        self.planted = set()  # planted positions of the whole block
        self.hist = set()  # touched positions before the current scan (far copy sources)

    def tpos(self, j: int) -> int:
        if j < 0:
            if self.e is None:
                raise Plan("no post-copy positions at the block start")
            return self.e + 1 + j
        return self.s + offs(j)

    def valid(self, j: int) -> bool:
        return self.tpos(j) + (1 if j < 0 else (32 + j) >> 5) <= self.limit

    def put(self, p: int, b: bytes):
        if p + len(b) > self.n:
            raise Plan("past the end")
        self.d[p:p + len(b)] = b

    def words(self, k: int):
        g = next(self.groups)
        return [g[i].to_bytes(4, "little") for i in range(k)]

    def plant(self, js, pattern):
        """Words at probe indices js; pattern: (group, member) per index: equal pairs are true repeats."""
        ps = [self.tpos(j) for j in js]
        if any(not self.valid(j) for j in js) or any(b - a < 4 for a, b in zip(ps, ps[1:])):
            raise Plan("plant does not fit")
        gw = {}
        for g, _ in pattern:
            if g not in gw:
                gw[g] = self.words(4)
        if js[0] == -2:  # the insert of ip-1: its first byte is the copy's last byte
            g0 = pattern[0][0]
            x = self.d[ps[0]]
            for grp in collisions(self.wm):
                firsts = [w for w in grp if w & 0xFF == x]
                if firsts:
                    ws = [w.to_bytes(4, "little") for w in [firsts[0]] + [w for w in grp if w != firsts[0]]]
                    gw[g0] = ws
                    break
            else:
                raise Plan("no word with that first byte")
        for p, (g, m) in zip(ps, pattern):
            if p == ps[0] and js[0] == -2:
                self.put(p + 1, gw[g][m][1:])
            else:
                self.put(p, gw[g][m])
            self.used.update(range(p, p + 4))
        self.touch += ps
        return ps

    def copy_at(self, j: int, q: int, ln: int):
        """Probe j hits candidate q (a position inserted earlier whose entry survives) and matches ln bytes."""
        p = self.tpos(j)
        if not self.valid(j) or q >= p or ln < 4 or p + ln > self.n:
            raise Plan("copy does not fit")
        for i in range(ln):
            self.d[p + i] = self.d[q + i]
        if p + ln < self.n and self.d[p + ln] == self.d[q + ln]:
            self.d[p + ln] ^= 0x5A
        if j == -1 and u32(self.d, p - 1) == u32(self.d, p):
            raise Plan("re-probe word equals the insert")
        self.copies.append((p, q, ln))
        self.ne = p + ln
        self.e, self.s = p + ln, p + ln + 1
        self.used = set()
        return p

    def source(self, j: int, off=None):
        """A filler probe position of this scan before index j (its word unique): a copy source."""
        cands = [self.tpos(i) for i in range(-2 if self.e is not None else 0, j)]
        cands = [q for q in cands if not (set(range(q, q + 4)) & self.used)]
        if not cands:
            raise Plan("no source")
        return cands[int(self.rng.integers(0, len(cands)))]

    def trigger(self, j: int, ln: int, q=None):
        p = self.tpos(j)
        if q is None:
            q = self.source(j)
        return self.copy_at(j, q, min(ln, self.n - p))

    def j_for_literal(self, lit: int) -> int:
        """Probe index whose position is next_emit + lit."""
        base = self.s - self.ne
        j = 0
        while base + offs(j) < lit:
            j += 1
        if base + offs(j) != lit:
            raise Plan("literal length not reachable here")
        return j


def _check(b: Builder, upto: int):
    tr = []
    d = bytes(b.d[: min(b.n, upto + 96)]) if upto + 96 + MARGIN < b.n else bytes(b.d)
    compress_fragment(d, b.wm, tr)
    cps = {(e[1], e[2], e[3]) for e in tr if e[0] == "c"}
    tps = {e[1] for e in tr if e[0] == "t"}
    ok = all(c in cps for c in b.copies) and all(p in tps for p in b.touch)
    n_c = sum(1 for e in tr if e[0] == "c")
    return ok and n_c == len(b.copies)


# ---------------------------------------------------------------------------------------- episodes
SHARE = {
    "pair": [(0, 0), (0, 1)],
    "triple": [(0, 0), (0, 1), (0, 2)],
    "quad": [(0, 0), (0, 1), (0, 2), (0, 3)],
    "AAB": [(0, 0), (0, 0), (0, 1)],
    "ABA": [(0, 0), (0, 1), (0, 0)],
    "BAA": [(0, 1), (0, 0), (0, 0)],
    "ABAB": [(0, 0), (1, 0), (0, 1), (1, 1)],   # interleaved pairs a < c < b < d
    "ABBA": [(0, 0), (1, 0), (1, 1), (0, 1)],   # nested pairs a < c < d < b
}
LIT_BEFORE = (1, 7, 31, 32, 33, 61, 63, 65, 127, 257)
COPY_LENS = (4, 5, 11, 12, 64, 65, 67, 68, 131, 132) + tuple(x for g in GS for x in (3 + g, 4 + g, 5 + g, 3 + 5 * g,
                                                                                      4 + 5 * g, 5 + 5 * g))


def ep_share(b: Builder, rng, strided=False):
    """A slot-sharing structure in one window: at the block start, behind a copy (j from -2), after a short copy in
    the window, or after 32 / 64 / 96 filler probes (strides 2, 3, 4, possibly across a stride change)."""
    kind = list(SHARE)[int(rng.integers(0, len(SHARE)))]
    pat = SHARE[kind]
    if strided:
        j = int(rng.choice([32, 64, 96])) + int(rng.integers(-6, 20))
        gap = max(1, 4 // ((32 + j) >> 5) + (1 if ((32 + j) >> 5) == 3 else 0))
        js = [j + gap * i + int(rng.integers(0, 3)) * i for i in range(len(pat))]
        js = sorted(set(js))
        if len(js) != len(pat):
            raise Plan("collapsed")
    else:
        lo = -2 if b.e is not None and rng.random() < 0.6 else 0
        span = int(rng.integers(4 * (len(pat) - 1), 32))
        cuts = sorted(rng.choice(np.arange(1, span), len(pat) - 2, replace=False).tolist()) if len(pat) > 2 else []
        rel = [0] + cuts + [span]
        rel = [rel[0]] + [max(r, rel[i] + 4) for i, r in enumerate(rel[1:])]
        js = [lo + r for r in rel]
        if js[-1] > 31:
            shift = js[-1] - 31
            js = [x - shift for x in js]
            if js[0] < lo:
                raise Plan("too wide")
    if kind in ("AAB", "BAA"):
        # a true repeat: the second copy of the word is a hit (a copy of 4 bytes); continue behind it
        i1 = pat.index((0, 0))
        i2 = pat.index((0, 0), i1 + 1)
        ps = b.plant(js[: i2 + 1], pat[: i2 + 1])
        q, p = ps[i1], ps[i2]
        if p + 4 < b.n and b.d[p + 4] == b.d[q + 4]:
            b.d[p + 4] ^= 0x33
        b.copies.append((p, q, 4))
        b.ne = p + 4
        b.e, b.s = p + 4, p + 5
        rest = pat[i2 + 1:]
        if rest:
            # behind the copy positions stay consecutive: -2 = p + 3, -1 = p + 4, j = p + 5 + j
            k = [b.e + 1 + (js[i2 + 1 + t] - js[i2]) - 5 for t in range(len(rest))]
            k = [max(x, -1) for x in k]
            g = b.words(2)
            for x, (_, m) in zip(k, rest):
                p2 = b.tpos(x)
                b.put(p2, g[m] if m else g[1])
                b.used.update(range(p2, p2 + 4))
                b.touch.append(p2)
        return kind
    b.plant(js, pat)
    return kind


def ep_pair_near(b: Builder, rng):
    """Two colliding, overlapping words 1-3 positions apart in a stride-1 window."""
    dist = int(rng.integers(1, 4))
    lo = -1 if b.e is not None and rng.random() < 0.5 else 0
    j = lo + int(rng.integers(0, 28))
    s = overlap_pairs(b.wm, dist)[int(rng.integers(0, 64))]
    p = b.tpos(j)
    if not b.valid(j + dist):
        raise Plan("end")
    b.put(p, s)
    b.used.update(range(p, p + len(s)))
    b.touch += [p, p + dist]
    return f"pair at {dist}"


def ep_trigger(b: Builder, rng, lit=None, ln=None):
    """End the scan with a copy: a chosen literal length in front of it and a chosen copy length."""
    if lit is None:
        lit = int(rng.choice(LIT_BEFORE)) if rng.random() < 0.5 else int(rng.integers(1, 34))
    if ln is None:
        ln = int(rng.choice(COPY_LENS)) if rng.random() < 0.6 else int(rng.integers(4, 12))
    base = b.s - b.ne
    if lit < base:
        lit = base
    j = b.j_for_literal(lit) if lit in reachable_literals() else b.j_for_literal(lit + 1)
    while b.tpos(j) in b.used or (set(range(b.tpos(j), b.tpos(j) + 4)) & b.used):
        j += 1
    b.trigger(j, ln)
    return "trigger"


def ep_short_copies(b: Builder, rng):
    """Short copies (4-8 bytes) that end inside the window, and chains of re-probe hits."""
    for _ in range(int(rng.integers(1, 4))):
        b.trigger(int(rng.integers(0 if b.e is None else -1, 6)), int(rng.integers(4, 9)))
    return "short copies"


def ep_skip_share(b: Builder, rng):
    """A copy skips a position whose word shares a slot with a probe behind the copy (the kernel's undo)."""
    j = int(rng.integers(12, 24))
    q = b.source(j - 8)
    x, y = b.words(2)
    b.put(q + 2, x)
    ln = int(rng.integers(7, 10))
    p = b.trigger(j, ln, q=q)
    k = int(rng.integers(0, 8))
    p2 = b.tpos(k)
    b.put(p2, y)
    b.used.update(range(p2, p2 + 4))
    b.touch.append(p2)
    return "skip share"


def ep_offset(b: Builder, rng, off):
    """A copy at a given offset: 1 (a byte run), 2, or far back to an earlier touched position."""
    if off <= 2:
        j = int(rng.integers(4, 20))
        p = b.tpos(j)
        x = int(rng.integers(0, 256))
        while x in b.runs:
            x = int(rng.integers(0, 256))
        b.runs.add(x)
        pat = bytes([x, (x + 1) & 0xFF]) if off == 2 else bytes([x])
        run = (pat * 40)[: 4 + off + int(rng.integers(0, 30))]
        b.put(p - off, run)
        if b.d[p - off - 1] == run[off - 1]:  # the run must not reach further back
            b.d[p - off - 1] ^= 0x77
        b.d[p - off + len(run)] = (run[len(run) - off] + 1) & 0xFF
        b.copies.append((p, p - off, len(run) - off))
        b.ne = p + len(run) - off
        b.e, b.s = b.ne, b.ne + 1
        b.used = set()
        return f"offset {off}"
    for j in range(0, 2000):
        if not b.valid(j):
            break
        q = b.tpos(j) - off
        if q in b.hist and q not in b.planted:
            return b.trigger(j, int(rng.choice((4, 11, 12, 40))), q=q) and f"offset {off}"
    raise Plan("no source at that offset")


def ep_cand0(b: Builder, rng):
    """The word at position 0 repeats at a probe whose slot was never written: candidate 0."""
    j = int(rng.integers(0, 40))
    b.trigger(j, int(rng.integers(4, 20)), q=0)
    return "candidate 0"


# ---------------------------------------------------------------------------------------- blocks
class Case:
    def __init__(self, data: bytes, name: str):
        self.data, self.name = data, name

    def __repr__(self):
        return f"Case({self.name}, {len(self.data)} B)"


def _history(b: Builder):
    tr = []
    compress_fragment(bytes(b.d[: b.n]), b.wm, tr)
    return {e[1] for e in tr if e[0] == "t" and e[1] < (b.e or 0)}


def build_block(seed: int, n: int, wm: int, theme: str, tokens=None, tail=None):
    """One block of n bytes at table size wm.  theme: "share" (slot sharing at every phase), "strided",
    "emit" (literal / copy lengths and offsets), "tokens" (exactly `tokens` copies), "end" (the scan end:
    tail = "none" | "last" | "limit" | "limit-1" | "n")."""
    rng = np.random.default_rng(seed)
    b = Builder(rng, n, wm)
    if n > 8192 and theme != "emit":
        # long blocks: a run of zeros (one copy at offset 1) and the episodes in the last 1.5-3.5 KiB
        h = n - int(rng.integers(1500, 3500))
        b.d[:h] = bytes(h)
        b.d[h] |= 1
        b.copies.append((1, 0, h - 1))
        b.ne = b.e = h
        b.s = h + 1
    reserve = 48 if theme != "tokens" else 0
    done = 0
    fails = 0
    while fails < 60:
        if tokens is not None and len(b.copies) >= tokens:
            break
        if b.s + 200 + reserve >= b.limit:
            break
        snap = (bytes(b.d), b.e, b.s, b.ne, set(b.used), list(b.copies), list(b.touch))
        try:
            if theme == "share":
                r = rng.random()
                if r < 0.55:
                    ep_share(b, rng)
                elif r < 0.75:
                    ep_pair_near(b, rng)
                elif r < 0.85:
                    ep_skip_share(b, rng)
                else:
                    ep_short_copies(b, rng)
                ep_trigger(b, rng, lit=None if rng.random() < 0.5 else int(rng.integers(34, 40)))
            elif theme == "strided":
                ep_share(b, rng, strided=True)
                ep_trigger(b, rng, lit=int(rng.integers(1 + offs(140), 1 + offs(150))))
            elif theme == "emit":
                r = rng.random()
                if r < 0.15 and wm >= 12:
                    b.hist = _history(b)
                    ep_offset(b, rng, int(rng.choice([2047, 2048, 2049, 4000, 16000])))
                elif r < 0.3:
                    ep_offset(b, rng, int(rng.integers(1, 3)))
                elif r < 0.37 and not b.copies:
                    ep_cand0(b, rng)
                else:
                    ep_trigger(b, rng, lit=int(rng.choice(LIT_BEFORE + (0,))) if rng.random() < 0.8 else None,
                               ln=int(rng.choice(COPY_LENS)))
            elif theme == "tokens":
                ep_trigger(b, rng, lit=int(rng.integers(1, 6)), ln=int(rng.integers(4, 9)))
            else:
                raise ValueError(theme)
            hi = max([c[0] + c[2] for c in b.copies] + b.touch + [0])
            if not _check(b, hi):
                raise Plan("the plan did not happen")
            b.planted.update(b.used)
            done += 1
        except (Plan, StopIteration, ValueError):
            b.d[:], b.e, b.s, b.ne, b.used, b.copies, b.touch = bytearray(snap[0]), *snap[1:5], snap[5], snap[6]
            fails += 1
    if tokens is not None and len(b.copies) != tokens:
        return None
    if theme == "end" or tail:
        _end(b, rng, tail)
    tr = []
    compress_fragment(bytes(b.d), wm, tr)
    if not _check(b, b.n):
        return None
    return Case(bytes(b.d), f"{theme} n={n} wm={wm} seed={seed}" + (f" tail={tail}" if tail else ""))


def _end(b: Builder, rng, tail):
    """Lay out the end of the block behind the last copy."""
    if tail in (None, "none"):
        return
    if tail == "last":
        # a copy such that the following scan's last valid probe (ip + step == ip_limit) hits
        for _ in range(400):
            p0 = b.s + int(rng.integers(0, 40))
            if p0 + 40 > b.limit:
                break
            e = p0 + int(rng.integers(4, 40))
            s, j = e + 1, 0
            while s + offs(j + 1) + ((32 + j + 1) >> 5) <= b.limit:
                j += 1
            if s + offs(j) + ((32 + j) >> 5) == b.limit and offs(j) > 8:
                jj = b.j_for_literal(p0 - b.ne) if p0 - b.ne in reachable_literals() else None
                if jj is None or b.tpos(jj) != p0:
                    continue
                b.trigger(jj, e - p0)
                b.copy_at(j, b.tpos(j - 1), 4)
                return
        raise Plan("no layout")
    target = tail if isinstance(tail, int) else {"limit": b.limit, "limit-1": b.limit - 1, "n": b.n}[tail]
    j = 0
    while b.valid(j + 1) and target - b.tpos(j + 1) >= 4:
        j += 1
    b.trigger(j, target - b.tpos(j))


@functools.lru_cache(maxsize=None)
def blocks(n: int, wm: int, count: int, seed: int = 0):
    """`count` generated blocks of n bytes for table size wm: every theme in turn (a failed layout is redrawn)."""
    themes = [("share", None, None), ("share", None, None), ("strided", None, None), ("emit", None, None),
              ("share", None, "none"), ("emit", None, "last"), ("share", None, "limit"), ("emit", None, "limit-1"),
              ("share", None, "n")]
    if 4096 <= n <= 8192:
        themes += [("tokens", k, None) for k in (31, 32, 33, 63, 64, 65)]
    out = []
    k = 0
    while len(out) < count:
        theme, tok, tail = themes[len(out) % len(themes)]
        c = None
        for attempt in range(8):
            k += 1
            try:
                c = build_block(seed * 7919 + 1000003 * wm + n + 31 * k, n, wm, theme, tokens=tok, tail=tail)
            except Plan:
                c = None
            if c is not None:
                break
        if c is None:
            raise RuntimeError(f"no layout for {theme} {tok} {tail} at n={n} wm={wm}")
        out.append(c)
    return out


def size_cases(seed: int = 5):
    """Short blocks (14-47 bytes: the 15-byte margin, one probe, the kernel's 16-byte staging granule) in random,
    repeating and constant forms; and final literals of every header boundary behind one copy."""
    rng = np.random.default_rng(seed)
    out = []
    for n in (14, 15, 16, 17, 18, 19, 20, 31, 32, 33, 47):
        out.append(Case(rng.integers(0, 256, n, dtype=np.uint8).tobytes(), f"random {n}"))
        out.append(Case(bytes(n), f"zero {n}"))
        w = rng.integers(0, 256, 5, dtype=np.uint8).tobytes()
        out.append(Case((w * 10)[:n], f"period 5, {n}"))
        out.append(Case(w[:1] + bytes(rng.integers(0, 256, 4, dtype=np.uint8)) + w[:4] * 3 +
                        rng.integers(0, 256, max(n - 17, 0), dtype=np.uint8).tobytes(), f"repeat at 1..5, {n}")
                   if n >= 17 else Case(bytes(n), f"zero {n}"))
    for k in range(32):
        # the last copy ends k + 1 bytes before ip_limit: the scan behind it runs into ip_limit after k + 2 touches
        for attempt in range(20):
            b = Builder(rng, 160, 13)
            try:
                _end(b, rng, b.limit - 1 - k)
            except Plan:
                continue
            if _check(b, b.n):
                out.append(Case(bytes(b.d), f"scan end after {k + 2} touches"))
                break
    for lit in (1, 32, 33, 60, 61, 62, 63, 64, 65, 127, 128, 129, 255, 256, 257, 258):
        # one copy near the start, then incompressible filler: the final literal is exactly `lit` bytes
        x = rng.integers(0, 256, 12, dtype=np.uint8).tobytes()
        head = x[:8] + x[:8]  # a hit at 8 (offset 8), copy up to the filler
        fill = rng.integers(0, 256, lit, dtype=np.uint8).tobytes()
        fill = bytes([fill[0] ^ (1 if fill[0] == head[8] else 0)]) + fill[1:] if lit else fill
        for pad in range(4):
            pre = rng.integers(0, 256, 8 * pad, dtype=np.uint8).tobytes()
            data = pre + head + fill
            tr = []
            compress_fragment(data, 13, tr)
            fin = [e for e in tr if e[0] == "l" and e[3]]
            if fin and fin[0][1] == lit:
                out.append(Case(data, f"final literal {lit}, op {fin[0][2] % 4}"))
    return out


# ---------------------------------------------------------------------------------------- coverage
EXT = sorted({x for g in GS for x in (3 + g, 4 + g, 5 + g, 3 + 5 * g, 4 + 5 * g, 5 + 5 * g)})
LIT_ALL = (1, 32, 33, 60, 61, 128, 129, 256, 257) + tuple(x for g in GS for x in (4 * g - 1, 4 * g + 1))
COPY_ALL = (4, 11, 12, 64, 65, 67, 68, 131, 132)
OFFSETS = (1, 2047, 2048, 2049)


def coverage(data: bytes, wm: int, counts=None):
    """Event classes of the serial parse of one block (defined on the reference's trace, not on the kernel's
    windows), added to the Counter `counts`:
    s1_share3     >= 3 touches on one slot among stride-1 touches spanning < 32 positions
    s1_repeat3    the same, with a true repeat among them (a hit) and a differing word
    aba           A-B-A on one slot: equal words around a colliding different one, within such a span
    interleaved / nested   two slots' pairs a < c < b < d / a < c < d < b within such a span
    pair_d<k>     two touches of one slot k positions apart within such a span
    postcopy_share   the insert of ip-1 or the re-probe of ip shares its slot with a touch < 32 positions on
    strided_share3   >= 3 touches on one slot within 32 consecutive probes of a scan, one at index >= 32
    skip_share    a copy skips a position whose word's slot is touched behind the copy within 32 positions
    lit_before_<L>, lit_final_<L>, lit_op<a>_<L>, copy_<L>, match_<m>, offset_<o>, tokens_<k>, tokens_mod32_0,
    room_cut, cand0, hit_last_probe, copy_end_limit, copy_end_limit-1, copy_end_n, scan_end_phase_<k>"""
    from collections import Counter
    c = Counter() if counts is None else counts
    tr = []
    compress_fragment(data, wm, tr)
    n = len(data)
    lim = n - MARGIN
    d = bytes(data) + bytes(4)
    T = [e for e in tr if e[0] == "t"]
    W = [u32(d, e[1]) for e in T]
    for i in range(len(T)):
        # stride-1 span starting at touch i
        span = []
        for k in range(i, len(T)):
            if T[k][3] >= 32 or T[k][1] - T[i][1] >= 32 or (k > i and T[k][1] <= T[k - 1][1]):
                break
            span.append(k)
        s0 = T[i][2]
        mine = [k for k in span if T[k][2] == s0]
        if len(mine) >= 3:
            c["s1_share3"] += 1
            ws = [W[k] for k in mine]
            if len(set(ws)) < len(ws) and len(set(ws)) > 1:
                c["s1_repeat3"] += 1
            for a in range(len(mine)):
                for b2 in range(a + 1, len(mine)):
                    for c2 in range(b2 + 1, len(mine)):
                        if W[mine[a]] == W[mine[c2]] != W[mine[b2]]:
                            c["aba"] += 1
        if len(mine) >= 2:
            c[f"pair_d{T[mine[1]][1] - T[i][1]}"] += 1
            if T[i][3] < 0:
                c["postcopy_share"] += 1
            b_ = mine[1]
            for k in span:
                if i < k < b_ and T[k][2] != s0:
                    other = [x for x in span if x > k and T[x][2] == T[k][2]]
                    if other:
                        c["interleaved" if other[0] > b_ else "nested"] += 1
                        break
        # strided: 32 consecutive probes of one scan
        if T[i][3] >= 0:
            run = [i]
            for k in range(i + 1, min(i + 32, len(T))):
                if T[k][3] != T[k - 1][3] + 1:
                    break
                run.append(k)
            same = [k for k in run if T[k][2] == s0]
            if len(same) >= 3 and any(T[k][3] >= 32 for k in same):
                c["strided_share3"] += 1
        if T[i][5] and T[i][3] >= 0 and T[i][1] + ((32 + T[i][3]) >> 5) == lim:
            c["hit_last_probe"] += 1
    slots_after = {}
    for e in T:
        slots_after.setdefault(e[2], []).append(e[1])
    cps = [e for e in tr if e[0] == "c"]
    for e in cps:
        _, ip, cand, m, op = e
        c[f"copy_{m}"] += 1
        c[f"match_{m}"] += 1
        c[f"offset_{ip - cand}"] += 1
        if ip + m == n:
            c["room_cut"] += 1
            c["copy_end_n"] += 1
        if ip + m == lim:
            c["copy_end_limit"] += 1
        if ip + m == lim - 1:
            c["copy_end_limit-1"] += 1
        if cand == 0:
            c["cand0"] += 1
        e_ = ip + m
        for x in range(ip + 1, e_ - 1):
            s = slot(u32(d, x), wm)
            if any(e_ - 1 <= p < ip + 32 for p in slots_after.get(s, ())):
                c["skip_share"] += 1
                break
    for e in tr:
        if e[0] == "l" and e[1]:
            c[f"lit_{'final' if e[3] else 'before'}_{e[1]}"] += 1
            c[f"lit_op{e[2] % 4}_{e[1]}"] += 1
    c[f"tokens_{len(cps)}"] += 1
    if cps and len(cps) % 32 == 0:
        c["tokens_mod32_0"] += 1
    # the last scan found nothing: its touches from the insert of ip-1 on, mod 32 (the kernel's lane phase)
    k = len(T)
    while k and T[k - 1][3] >= 0 and not T[k - 1][5]:
        k -= 1
    if n >= MARGIN and (not T or not T[-1][5]):
        c[f"scan_end_phase_{(len(T) - k + (2 if k else 0)) % 32}"] += 1
    return c


@functools.lru_cache(maxsize=None)
def corpus(wm: int):
    """The generated blocks for table size wm: 18 of 4 KiB, 9 of 32 KiB (the GPU and CPU conformance tests)."""
    return blocks(4096, wm, 18) + blocks(32768, wm, 9)
