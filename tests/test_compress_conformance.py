"""The Python restatement of csnappy_compress_fragment (tests/compress_cases.py) against the oracle port, and the
coverage of the generated compressor blocks.

The GPU compressor tests compare the kernel with the oracle on these blocks; that is only worth something if the
blocks drive the parse through the cases the kernel treats specially.  The coverage assertions below are defined
on the reference's serial trace (not on the kernel's windows), and every structure is planted at several phases, so
whichever windows the kernel forms, some of them hold it."""
import os
import sys
from collections import Counter

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import compress_cases as CC  # noqa: E402
import oracle  # noqa: E402
from cases import EDGE_FRAGMENT_SIZES, fuzz_pages  # noqa: E402

WMS = (9, 13, 15, 16)


@pytest.fixture(scope="module")
def port():
    return oracle.port()


@pytest.mark.parametrize("wm", WMS)
def test_restatement_equals_port_on_generated_blocks(port, wm):
    for c in CC.corpus(wm):
        assert CC.compress_fragment(c.data, wm) == port.compress_fragment(c.data, wm), c.name
    for c in CC.size_cases():
        assert CC.compress_fragment(c.data, wm) == port.compress_fragment(c.data, wm), c.name


def test_restatement_equals_port_on_existing_corpora(port, urls):
    # the sizes and table sizes of test_gpu_parity.py::test_batch_compress_fuzz_vs_oracle (every 4th page)
    for size, wm in ((4096, 13), (4096, 9), (32768, 15), (32768, 16), (1000, 12), (20000, 14), (64, 10)):
        for p in fuzz_pages(4321 + size + wm, 70, size)[::4]:
            assert CC.compress_fragment(p, wm) == port.compress_fragment(p, wm), (size, wm)
    for block, wm in ((4096, 13), (32768, 15), (4096, 9)):
        for o in range(0, min(len(urls), 200000), block * 5):
            assert CC.compress_fragment(urls[o:o + block], wm) == port.compress_fragment(urls[o:o + block], wm)
    text = urls[:40000]
    for n in EDGE_FRAGMENT_SIZES:
        for wm in (9, 16):
            assert CC.compress_fragment(text[:n], wm) == port.compress_fragment(text[:n], wm), n


def test_literal_lengths_before_a_copy_are_probe_distances(urls):
    """A copy starts at a probe position, so the literal in front of it is 0 or 1 + a distance of the skip
    schedule: 60, 128, 129 and 256 never precede a copy (the kernel's header-size paths for those lengths are
    reached by final literals only)."""
    reach = CC.reachable_literals()
    assert not {60, 128, 129, 256} & reach and {1, 32, 33, 61, 63, 65, 127, 257} <= reach
    for wm in (9, 13):
        tr = []
        for c in CC.corpus(wm)[:10]:
            CC.compress_fragment(c.data, wm, tr)
        for o in range(0, 300000, 32768):
            CC.compress_fragment(urls[o:o + 32768], wm, tr)
        assert all(e[1] in reach for e in tr if e[0] == "l" and not e[3])


# (event class, at least this many in the 4 KiB blocks, in the 32 KiB blocks), per table size
NEED = [
    ("s1_share3", 20, 10), ("s1_repeat3", 5, 5), ("aba", 3, 2), ("interleaved", 10, 10), ("nested", 10, 10),
    ("postcopy_share", 50, 50), ("strided_share3", 2, 1), ("skip_share", 10, 5),
    ("hit_last_probe", 1, 1), ("copy_end_limit", 1, 1), ("copy_end_limit-1", 1, 1), ("copy_end_n", 1, 1),
    ("offset_1", 20, 20), ("tokens_mod32_0", 1, 0),
] + [(f"pair_d{k}", 1, 1) for k in range(1, 32)] + [(f"copy_{m}", 1, 1) for m in CC.COPY_ALL] + \
    [(f"match_{m}", 1, 1) for m in CC.EXT] + \
    [(f"lit_before_{L}", 3, 3) for L in CC.LIT_ALL if L in CC.reachable_literals()] + \
    [(f"tokens_{k}", 1, 0) for k in (31, 32, 33, 63, 64, 65)]


@pytest.mark.parametrize("wm", WMS)
def test_generated_blocks_cover_every_event_class(wm):
    for n, col in ((4096, 1), (32768, 2)):
        cnt = Counter()
        for c in CC.corpus(wm):
            if len(c.data) == n:
                CC.coverage(c.data, wm, cnt)
        missing = [(k, cnt[k], need[col]) for need in NEED for k in [need[0]] if cnt[k] < need[col]]
        assert not missing, (n, wm, missing)
        if wm >= 13:  # (at wm 9 the source's slot is overwritten long before)
            offs = [cnt[f"offset_{o}"] for o in (2047, 2048, 2049)]
            assert (all(offs) if n == 32768 else sum(offs)), (n, wm, offs)
        if n == 32768:
            assert cnt["cand0"] >= 1
        # literals at every output alignment in front of copies
        assert all(cnt[f"lit_op{a}_{L}"] for a in range(4) for L in (1, 32, 33)), (n, wm)
        assert sum(1 for k in range(32) if cnt[f"scan_end_phase_{k}"]) >= 4, (n, wm)


def test_size_cases_cover_final_literals_and_scan_end_phases():
    cnt = Counter()
    for c in CC.size_cases():
        CC.coverage(c.data, 13, cnt)
    for L in (32, 33, 60, 61, 128, 129, 256, 257, 63, 65, 127):
        assert cnt[f"lit_final_{L}"] >= 1, L
    # a scan that runs into ip_limit without a hit, at every lane phase
    assert all(cnt[f"scan_end_phase_{k}"] for k in range(32)), [k for k in range(32) if not cnt[f"scan_end_phase_{k}"]]
