"""Pin the oracle (oracle/snappy_oracle.c) before anything trusts it.

Two anchors (SURVEY.md 8c), both committed under tests/golden/ (tests/golden/make_golden.py):
  1. golden.json: the unmodified reference on its own fixtures and on seeded synthetic inputs;
  2. reference_cases.json: the results on the fuzz, edge-size and corrupted-stream inputs of
     tests/cases.py that these tests compared with the compiled reference.  Its `checker` names
     what recorded them: the port, unchanged since it was compared with the reference on them.
Mirrors the reference's own checks: round trip of urls.10K (Makefile:21-27),
`cl_tester -S d` error codes (cl_tester.c:167-238), baddata3 (Makefile:33),
unaligned_uint64 (Makefile:37-55).
"""
import hashlib
import struct

import numpy as np
import pytest

import oracle
from cases import (EDGE_COMPRESS_SIZES, EDGE_FRAGMENT_SIZES, corrupted_fragments, edge_compress_input, edge_text,
                   ends_inside_tag, fuzz_pages, reference_cases, synth_cases)


def sha(b):
    return hashlib.sha256(b).hexdigest()


@pytest.fixture(scope="module")
def port():
    return oracle.port()


def test_fixture_integrity(golden, urls, urls_snappy, baddata3, unaligned_pair):
    fx = golden["fixtures"]
    assert sha(urls) == fx["urls.10K"]["sha256"]
    assert sha(urls_snappy) == fx["urls.10K.snappy"]["sha256"]
    assert sha(baddata3) == fx["baddata3.snappy"]["sha256"]
    assert sha(unaligned_pair[0]) == fx["unaligned_uint64_test.snappy"]["sha256"]
    assert sha(unaligned_pair[1]) == fx["unaligned_uint64_test.bin"]["sha256"]


def test_compress_urls_wm15_is_the_checked_in_fixture(port, urls, urls_snappy):
    assert port.compress(urls, 15) == urls_snappy


@pytest.mark.parametrize("wm", range(9, 17))
def test_compress_urls_all_table_sizes(port, golden, urls, wm):
    c = port.compress(urls, wm)
    g = golden["compress_urls"][str(wm)]
    assert len(c) == g["len"] and sha(c) == g["sha256"]


@pytest.mark.parametrize("key", ["4096/13", "32768/15", "32768/16", "4096/9", "4096/16"])
def test_fragment_streams(port, golden, urls, key):
    block, wm = map(int, key.split("/"))
    parts, total = [], 0
    for o in range(0, len(urls), block):
        c = port.compress_fragment(urls[o:o + block], wm)
        parts.append(struct.pack("<I", len(c)) + c)
        total += len(c)
    g = golden["fragments_urls"][key]
    assert (len(parts), total, sha(b"".join(parts))) == (g["blocks"], g["total"], g["sha256"])


def test_tiny_inputs(port, golden):
    for label, g in golden["tiny"].items():
        assert port.compress(bytes.fromhex(g["input_hex"]), 16).hex() == g["wm16_hex"], label


def test_synth_cases_vs_golden(port, golden):
    for name, data in synth_cases().items():
        g = golden["synth"][name]
        assert sha(data) == g["in_sha256"], name
        for wm in (9, 13, 15, 16):
            c = port.compress_fragment(data, wm)
            assert (len(c), sha(c)) == (g[f"frag_wm{wm}"]["len"], g[f"frag_wm{wm}"]["sha256"]), (name, wm)
            rc, back = port.decompress_noheader(c, len(data))
            assert rc == 0 and back == data, (name, wm)


def test_decode_matrix_noheader(port, golden):
    for e in golden["decode_noheader"]:
        rc, out = port.decompress_noheader(bytes.fromhex(e["hex"]), e["cap"])
        assert rc == e["rc"], e
        if rc == 0:
            assert out.hex() == e["out_hex"], e


def test_decode_matrix_header(port, golden):
    for e in golden["decode_header"]:
        rc, _ = port.decompress(bytes.fromhex(e["hex"]), e["dst_len"])
        assert rc == e["rc"], e


def test_varint(port, golden):
    for e in golden["varint"]:
        rc, val = port.get_uncompressed_length(bytes.fromhex(e["hex"]))
        assert rc == e["rc"], e
        if rc > 0:
            assert val == e["value"], e


def test_truncated_tags_are_malformed(port):
    # copy-1 / copy-2 / copy-4 / long literal whose trailing bytes are cut off: -5 by definition
    for hx in ("0861626301", "0861626302", "086162630203", "086162630f0300", "f0", "f4ff"):
        rc, _ = port.decompress_noheader(bytes.fromhex(hx), 100)
        assert rc == oracle.E_DATA_MALFORMED, hx


def test_roundtrip_urls(port, urls, urls_snappy):
    rc, out = port.decompress(urls_snappy, len(urls))
    assert rc == 0 and out == urls
    assert port.get_uncompressed_length(urls_snappy) == (3, len(urls))
    # too-small destination => -2 ; noheader with small capacity => -3 (cl_tester.c:196-218)
    assert port.decompress(urls_snappy, 4096)[0] == oracle.E_OUTPUT_INSUF
    assert port.decompress_noheader(urls_snappy[3:], 4096)[0] == oracle.E_OUTPUT_OVERRUN


def test_baddata3(port, golden, baddata3):
    rc, _ = port.decompress(baddata3, golden["baddata3"]["header_len"])
    assert rc == golden["baddata3"]["rc"] == oracle.E_DATA_MALFORMED


def test_unaligned_uint64(port, golden, unaligned_pair):
    comp, expect = unaligned_pair
    rc, out = port.decompress(comp, len(expect))
    assert rc == 0 and out == expect and sha(out) == golden["unaligned_uint64"]["out_sha256"]


def test_chunk_table_rule(port):
    # csnappy_compress.c:638-646
    assert port.chunk_wm(32768, 16) == 16
    assert port.chunk_wm(4096, 16) == 13
    assert port.chunk_wm(4097, 16) == 14
    assert port.chunk_wm(13959, 15) == 15
    assert port.chunk_wm(13959, 16) == 15
    assert port.chunk_wm(1, 16) == 9
    assert port.chunk_wm(300, 9) == 9


@pytest.mark.parametrize("size,wm", [(4096, 13), (4096, 9), (32768, 15), (32768, 16), (1000, 12), (20000, 14)])
def test_port_equals_reference_on_fuzz(port, size, wm):
    want = reference_cases()["fuzz_fragments"][f"{size}/{wm}"]
    pages = fuzz_pages(1234 + size + wm, 35, size)
    assert len(pages) == len(want)
    for i, page in enumerate(pages):
        a = port.compress_fragment(page, wm)
        assert sha(a) == want[i], (i, size, wm)
        assert port.decompress_noheader(a, size) == (0, page)


def test_port_equals_reference_on_edge_sizes(port):
    ref = reference_cases()
    text = edge_text()
    for wm in (9, 13, 16):
        for n, want in zip(EDGE_FRAGMENT_SIZES, ref["edge_fragments"][str(wm)], strict=True):
            assert sha(port.compress_fragment(text[:n], wm)) == want, (n, wm)
    for wm in (9, 13, 15, 16):
        for n, want in zip(EDGE_COMPRESS_SIZES, ref["edge_compress"][str(wm)], strict=True):
            assert sha(port.compress(edge_compress_input(text, n), wm)) == want, (n, wm)


def test_port_decoder_equals_reference_on_corruptions(port):
    """Flip / truncate valid streams; both decoders must agree on rc and, on success, on bytes.
    Streams whose LAST tag is cut inside its trailing bytes are skipped: that case is undefined
    behaviour in the reference's x86 path (SURVEY.md 0.5) and defined as -5 here."""
    checked = 0
    for (d, cap), want in zip(corrupted_fragments(port.compress_fragment), reference_cases()["corruptions"], strict=True):
        rc, out = port.decompress_noheader(d, cap)
        if rc == oracle.E_DATA_MALFORMED and ends_inside_tag(d):
            continue
        assert [rc, None if out is None else sha(out)] == want, (d.hex(), cap)
        checked += 1
    assert checked > 500


def test_bulk_harness_port_vs_reference():
    want = reference_cases()["bulk_4096_13"]
    pages = np.frombuffer(b"".join(fuzz_pages(77, 64, 4096)), dtype=np.uint8).reshape(64, 4096)
    o1, l1, _ = oracle.batch_compress(pages, 13, "port", threads=2)
    o2, l2, _ = oracle.batch_compress(pages, 13, "port", threads=3)
    assert l1.tolist() == l2.tolist() == want["len"]
    for i in range(64):
        assert sha(o1[i, : l1[i]].tobytes()) == sha(o2[i, : l2[i]].tobytes()) == want["sha256"][i], i
    d1, n1, s1, _ = oracle.batch_decompress(o1, l1, 4096, "port", threads=2)
    d2, n2, s2, _ = oracle.batch_decompress(o2, l2, 4096, "port", threads=1)
    assert (s1 == 0).all() and (s2 == 0).all() and (n1 == 4096).all() and (n2 == 4096).all()
    assert (d1[:, :4096] == pages).all() and (d2[:, :4096] == pages).all()


def test_batch_runner_is_the_bench_cpu_protocol():
    """oracle.BatchRunner (bench.py's one CPU-baseline protocol): buffers allocated once, compress + decompress timed in
    the C harness, exact round trip, and the same bytes as the single-block entry points."""
    pages = fuzz_pages(31, 200, 4096)
    units = np.frombuffer(b"".join(pages), dtype=np.uint8).reshape(len(pages), 4096)
    for impl in (["reference"] if oracle.have_reference() else []) + ["port"]:
        r = oracle.BatchRunner(units, 13, impl, threads=3)
        tc, td = r.measure(warmup=1, steps=2)
        assert tc > 0 and td > 0
        chk = oracle.reference() if impl == "reference" else oracle.port()
        for i in (0, 57, 199):
            assert r.compressed(i) == chk.compress_fragment(pages[i], 13)
