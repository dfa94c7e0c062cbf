"""GPU parity tests: the CUDA path, called through the C-ABI (ctypes), against the oracle.

Bit-exact bar: compressed bytes, produced bytes, lengths and return codes must be
identical to the oracle's (the unmodified reference when oracle/_ref was built, else
our pinned restatement) and to the committed golden vectors.  Mirrors the reference's
own checks: `make cl_test` (Makefile:21-29), cl_tester -S d (cl_tester.c:167-238),
baddata3 (Makefile:33), check_unaligned_uint64 (Makefile:37-55).
"""
import hashlib
import struct

import numpy as np
import pytest

import oracle
from cases import fuzz_pages, synth_cases
from containers import ref_container

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def sha(b):
    return hashlib.sha256(b).hexdigest()


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.fixture(scope="module")
def chk():
    return oracle.best()


# --------------------------------------------------------------------------- drop-in API (host pointers)
def test_dropin_compress_urls_wm15_equals_fixture(cs, urls, urls_snappy):
    assert cs.csnappy_compress(urls, 15) == urls_snappy


@pytest.mark.parametrize("wm", range(9, 17))
def test_dropin_compress_urls_all_wm(cs, golden, urls, wm):
    c = cs.csnappy_compress(urls, wm)
    g = golden["compress_urls"][str(wm)]
    assert (len(c), sha(c)) == (g["len"], g["sha256"])


def test_dropin_roundtrip_urls(cs, urls, urls_snappy):
    rc, out = cs.csnappy_decompress(urls_snappy, len(urls))
    assert rc == 0 and out == urls
    c16 = cs.csnappy_compress(urls, 16)
    rc, out = cs.csnappy_decompress(c16, len(urls))
    assert rc == 0 and out == urls


def test_dropin_selftest_decompression(cs, chk):
    """cl_tester.c:167-238: -2 on small dst, -3 from noheader with small capacity, cut literal != OK."""
    rng = np.random.default_rng(1)
    data = rng.integers(0, 256, 4096 + 100, dtype=np.uint8).tobytes()
    comp = cs.csnappy_compress(data, 16)
    assert comp == chk.compress(data, 16)
    assert cs.csnappy_decompress(comp, 4096)[0] == cs.CSNAPPY_E_OUTPUT_INSUF
    hlen, n = cs.csnappy_get_uncompressed_length(comp)
    assert hlen > 0 and n == len(data)
    assert cs.csnappy_decompress_noheader(comp[hlen:], 4096)[0] == cs.CSNAPPY_E_OUTPUT_OVERRUN
    fake = bytes.fromhex("32c4666f6f6f6f6f6f")
    assert cs.csnappy_decompress(fake, 50)[0] == cs.CSNAPPY_E_DATA_MALFORMED
    assert cs.csnappy_decompress_noheader(fake[1:], 50)[0] == cs.CSNAPPY_E_DATA_MALFORMED


def test_dropin_baddata3(cs, golden, baddata3):
    rc, _ = cs.csnappy_decompress(baddata3, golden["baddata3"]["header_len"])
    assert rc == golden["baddata3"]["rc"] == -5


def test_dropin_unaligned_uint64(cs, unaligned_pair):
    comp, expect = unaligned_pair
    rc, out = cs.csnappy_decompress(comp, len(expect))
    assert rc == 0 and out == expect


def test_dropin_decode_matrix(cs, golden):
    for e in golden["decode_noheader"]:
        rc, out = cs.csnappy_decompress_noheader(bytes.fromhex(e["hex"]), e["cap"])
        assert rc == e["rc"], e
        if rc == 0:
            assert out.hex() == e["out_hex"], e
    for e in golden["decode_header"]:
        assert cs.csnappy_decompress(bytes.fromhex(e["hex"]), e["dst_len"])[0] == e["rc"], e
    for hx in ("0861626301", "0861626302", "086162630203", "086162630f0300", "f0", "f4ff"):
        assert cs.csnappy_decompress_noheader(bytes.fromhex(hx), 100)[0] == -5, hx


def test_dropin_tiny_and_synth(cs, golden):
    for label, g in golden["tiny"].items():
        assert cs.csnappy_compress(bytes.fromhex(g["input_hex"]), 16).hex() == g["wm16_hex"], label
    for name, data in synth_cases().items():
        g = golden["synth"][name]
        for wm in (9, 13, 15, 16):
            c = cs.csnappy_compress_fragment(data, wm)
            assert (len(c), sha(c)) == (g[f"frag_wm{wm}"]["len"], g[f"frag_wm{wm}"]["sha256"]), (name, wm)
            assert cs.csnappy_decompress_noheader(c, len(data)) == (0, data), (name, wm)


def test_dropin_multichunk_sizes(cs, chk):
    rng = np.random.default_rng(3)
    text = bytes(rng.integers(97, 101, 200000, dtype=np.uint8))
    for n in (0, 1, 14, 15, 32767, 32768, 32769, 65536, 70001, 150000):
        for wm in (9, 13, 16):
            c = cs.csnappy_compress(text[:n], wm)
            assert c == chk.compress(text[:n], wm), (n, wm)
            assert cs.csnappy_decompress(c, n) == (0, text[:n])


# --------------------------------------------------------------------------- device batches
def _to_dev(pages, stride):
    B = len(pages)
    host = np.zeros((B, stride), dtype=np.uint8)
    lens = np.zeros(B, dtype=np.int32)
    for i, p in enumerate(pages):
        host[i, : len(p)] = np.frombuffer(p, dtype=np.uint8)
        lens[i] = len(p)
    return torch.from_numpy(host).cuda(), torch.from_numpy(lens).cuda(), host, lens


def _gpu_compress(cs, pages, block, wm, lanes=0, var_len=False):
    """lanes: 0 / 8 / 16 / 32 = lane group (block staged in shared memory as the launcher decides);
    -32 = 32-lane groups reading the block from global memory (the form large fragments take in large batches)"""
    cs.set_tuning("compress_stage_input", 2 if lanes < 0 else 0)
    cs.set_tuning("compress_lanes", abs(lanes))
    try:
        d_in, d_len, _, _ = _to_dev(pages, block)
        out, out_len = cs.batch_compress_fragments(d_in, block, len(pages), wm, in_len=d_len if var_len else None)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("compress_lanes", 0)
        cs.set_tuning("compress_stage_input", 0)
    ostride = cs.api.out_stride_for(block)
    o = out.cpu().numpy().reshape(-1)[: len(pages) * ostride].reshape(len(pages), ostride)
    ln = out_len.cpu().numpy().astype(np.uint32)
    return [o[i, : ln[i]].tobytes() for i in range(len(pages))], out, out_len


@pytest.mark.parametrize("lanes", [32, 16, 8, -32])
@pytest.mark.parametrize("key", ["4096/13", "32768/15", "32768/16", "4096/9", "4096/16"])
def test_batch_compress_urls_fragments(cs, golden, urls, key, lanes):
    block, wm = map(int, key.split("/"))
    pages = [urls[o:o + block] for o in range(0, len(urls), block)]
    comp, _, _ = _gpu_compress(cs, pages, block, wm, lanes, var_len=True)
    stream = b"".join(struct.pack("<I", len(c)) + c for c in comp)
    g = golden["fragments_urls"][key]
    assert (len(comp), sum(map(len, comp)), sha(stream)) == (g["blocks"], g["total"], g["sha256"])


@pytest.mark.parametrize("lanes", [32, 16, 8, -32])
@pytest.mark.parametrize("size,wm", [(4096, 13), (4096, 9), (32768, 15), (32768, 16), (1000, 12), (20000, 14), (64, 10)])
def test_batch_compress_fuzz_vs_oracle(cs, chk, size, wm, lanes):
    pages = fuzz_pages(4321 + size + wm, 70, size)
    comp, _, _ = _gpu_compress(cs, pages, size, wm, lanes)
    for i, (p, c) in enumerate(zip(pages, comp)):
        assert c == chk.compress_fragment(p, wm), (i, size, wm, lanes)


def test_batch_compress_edge_sizes(cs, chk):
    rng = np.random.default_rng(7)
    text = bytes(rng.integers(97, 101, 40000, dtype=np.uint8))
    sizes = list(range(0, 40)) + [59, 60, 61, 62, 255, 256, 257, 258] + list(range(4081, 4112)) + list(range(32753, 32769))
    pages = [text[:n] for n in sizes]
    for wm, lanes in ((9, 0), (13, 0), (16, 0), (13, -32), (15, -32)):
        comp, _, _ = _gpu_compress(cs, pages, 32768, wm, lanes, var_len=True)
        for n, c in zip(sizes, comp):
            assert c == chk.compress_fragment(text[:n], wm), (n, wm, lanes)


def test_batch_compress_shrink_table_flag(cs, chk):
    rng = np.random.default_rng(8)
    text = bytes(rng.integers(97, 103, 32768, dtype=np.uint8))
    sizes = [100, 255, 256, 257, 4096, 4097, 13959, 32767, 32768]
    d_in, d_len, _, _ = _to_dev([text[:n] for n in sizes], 32768)
    out, out_len = cs.batch_compress_fragments(d_in, 32768, len(sizes), 16, in_len=d_len, flags=cs.api.BATCH_SHRINK_TABLE)
    torch.cuda.synchronize()
    ostride = cs.api.out_stride_for(32768)
    o = out.cpu().numpy()
    for i, n in enumerate(sizes):
        got = o[i * ostride: i * ostride + int(out_len[i])].tobytes()
        assert got == chk.compress_fragment(text[:n], oracle.port().chunk_wm(n, 16)), n


@pytest.mark.parametrize("stage", [0, 2, 4])
@pytest.mark.parametrize("lanes", [32, 16, 8])
def test_batch_decompress_roundtrip_and_errors(cs, chk, lanes, stage):
    pages = fuzz_pages(99, 140, 4096)
    comp = [chk.compress_fragment(p, 13) for p in pages]
    rng = np.random.default_rng(5)
    streams, caps = [], []
    for i, c in enumerate(comp):
        d = bytearray(c)
        k = i % 5
        if k == 1 and len(d) > 8:
            d[int(rng.integers(0, len(d)))] ^= int(rng.integers(1, 256))
        elif k == 2 and len(d) > 8:
            d = d[: int(rng.integers(1, len(d)))]
        streams.append(bytes(d))
        caps.append(4096 if k != 3 else 2000)
    stride = cs.csnappy_max_compressed_length(4096) + 6
    stride = (stride + 15) // 16 * 16
    d_in, d_len, _, _ = _to_dev(streams, stride)
    d_caps = torch.tensor(caps, dtype=torch.int32).cuda()
    cs.set_tuning("decompress_lanes", lanes)
    cs.set_tuning("decompress_stage_input", stage)
    try:
        out, out_len, status = cs.batch_decompress(d_in, d_len, len(streams), 4096, in_stride=stride, out_caps=d_caps,
                                                   out_stride=4096)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("decompress_lanes", 0)
        cs.set_tuning("decompress_stage_input", 0)
    o, ol, st = out.cpu().numpy(), out_len.cpu().numpy(), status.cpu().numpy()
    n_err = 0
    for i, s in enumerate(streams):
        rc, exp = oracle.port().decompress_noheader(s, caps[i])  # the port defines the truncated-tag case as -5
        assert st[i] == rc, (i, s.hex()[:80])
        if rc == 0:
            assert ol[i] == len(exp) and o[i * 4096: i * 4096 + ol[i]].tobytes() == exp, i
        else:
            n_err += 1
            assert ol[i] == 0
    assert n_err > 20


@pytest.mark.parametrize("stage", [0, 4])
def test_batch_decompress_with_header_and_streaming_path(cs, chk, urls, urls_snappy, baddata3, unaligned_pair, stage):
    """Whole multi-chunk streams in one batch: exercises the global-memory path (stage 0: a warp per stream,
    stage 4: a lane per stream) and -1/-2."""
    uu_s, uu_b = unaligned_pair
    streams = [urls_snappy, baddata3, uu_s, b"", bytes.fromhex("80"), chk.compress(urls[:5000], 16), urls_snappy]
    caps = [len(urls), 130378, len(uu_b), 10, 10, 5000, 4096]
    expect_rc = [0, -5, 0, -1, -1, 0, -2]
    off = np.zeros(len(streams), dtype=np.int64)
    pos = 0
    for i, s in enumerate(streams):
        off[i] = pos
        pos += (len(s) + 15) // 16 * 16 + 16
    host = np.zeros(pos, dtype=np.uint8)
    for i, s in enumerate(streams):
        host[off[i]: off[i] + len(s)] = np.frombuffer(s, dtype=np.uint8)
    d_in = torch.from_numpy(host).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_len = torch.tensor([len(s) for s in streams], dtype=torch.int32).cuda()
    d_caps = torch.tensor(caps, dtype=torch.int32).cuda()
    ostride = (max(caps) + 15) // 16 * 16
    cs.set_tuning("decompress_stage_input", stage)
    try:
        out, out_len, status = cs.batch_decompress(d_in, d_len, len(streams), 0, in_off=d_off, out_caps=d_caps,
                                                   out_stride=ostride, flags=cs.api.BATCH_WITH_HEADER)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("decompress_stage_input", 0)
    st, ol, o = status.cpu().numpy(), out_len.cpu().numpy(), out.cpu().numpy()
    assert list(st) == expect_rc
    assert o[: ol[0]].tobytes() == urls
    assert o[2 * ostride: 2 * ostride + ol[2]].tobytes() == uu_b
    assert o[5 * ostride: 5 * ostride + ol[5]].tobytes() == urls[:5000]


def test_batch_pack(cs):
    rng = np.random.default_rng(11)
    n, stride = 1000, 4816
    lens = rng.integers(0, 4811, n).astype(np.int32)
    lens[:5] = [0, 1, 3, 4810, 17]
    slots = rng.integers(0, 256, (n, stride), dtype=np.uint8)
    d_slots = torch.from_numpy(slots).cuda()
    d_len = torch.from_numpy(lens).cuda()
    packed, off = cs.batch_pack(d_slots, stride, d_len, n)
    torch.cuda.synchronize()
    off = off.cpu().numpy()
    assert (off[:-1] == np.concatenate([[0], np.cumsum(lens.astype(np.int64))[:-1]])).all() and off[-1] == lens.sum()
    p = packed.cpu().numpy()
    for i in range(n):
        assert (p[off[i]: off[i] + lens[i]] == slots[i, : lens[i]]).all(), i


def test_c_caller_through_the_plain_c_abi(cs, urls, urls_snappy, tmp_path):
    """tests/c/dropin_main.c: cl_tester / zram / block_compressor style calls from C."""
    import subprocess

    from test_cabi import build_c_caller

    exe = build_c_caller(tmp_path)
    a, b = tmp_path / "urls.10K", tmp_path / "urls.10K.snappy"
    a.write_bytes(urls)
    b.write_bytes(urls_snappy)
    r = subprocess.run([exe, str(a), str(b)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "dropin ok" in r.stdout, r.stdout + r.stderr


# --------------------------------------------------------------------------- block_compressor container
@pytest.mark.parametrize("page,wm", [(4096, 13), (1024, 11), (32768, 15)])
def test_bc_container_matches_reference_writer_and_round_trips(cs, chk, urls, page, wm):
    rng = np.random.default_rng(21)
    data = (urls[:150000] + rng.integers(0, 256, 3 * page + 17, dtype=np.uint8).tobytes() + bytes(5 * page) +
            urls[150000:150000 + 2 * page + 1234])
    h_in = np.frombuffer(data, dtype=np.uint8).copy()
    cont = np.zeros(cs.api.bc_max_container_length(len(data), page), dtype=np.uint8)
    clen = cs.api.bc_compress_host(h_in, len(data), cont, wm, page)
    ref = ref_container(chk, data, page, wm)
    assert clen == len(ref) and cont[:clen].tobytes() == ref
    nr = (len(data) + page - 1) // page
    out = np.zeros(nr * page, dtype=np.uint8)
    rc, olen, bad = cs.api.bc_decompress_host(cont, clen, out, page)
    assert (rc, olen, bad) == (0, len(data), None) and out[:olen].tobytes() == data


def test_bc_container_many_chunks_and_errors(cs, chk):
    """More pages than one pipeline chunk (8192 x 4 KiB), then corrupt / truncated containers."""
    from csnappy_b200 import synth

    B, page = 20000, 4096
    h_in = synth.mixed_pages(B, page, seed=77, device="cuda", pool_bytes=1 << 20).cpu().numpy()
    cont = np.zeros(cs.api.bc_max_container_length(B * page, page), dtype=np.uint8)
    clen = cs.api.bc_compress_host(h_in, B * page, cont, 13, page)
    idx = cont[4:4 + 4 * B].view(np.uint32)
    ref_out, ref_len, _ = oracle.batch_compress(h_in.reshape(B, page), 13, chk.kind, threads=4)
    want = np.minimum(ref_len, page)
    assert int(cont[:4].view(np.uint32)[0]) == B and (idx == want).all() and clen == 4 + 4 * B + int(want.sum())
    off = 4 + 4 * B + np.concatenate([[0], np.cumsum(want.astype(np.int64))])
    for i in list(range(0, B, 997)) + [B - 1]:
        exp = h_in[i * page:(i + 1) * page] if ref_len[i] >= page else ref_out[i, : ref_len[i]]
        assert (cont[off[i]: off[i + 1]] == exp).all(), i
    out = np.zeros(B * page, dtype=np.uint8)
    rc, olen, bad = cs.api.bc_decompress_host(cont, clen, out, page)
    assert (rc, olen, bad) == (0, B * page, None) and (out == h_in).all()
    # corrupt one compressed page (first text page after page 9000): its decode must fail or differ, never crash
    victim = next(i for i in range(9000, B) if 100 < idx[i] < page)
    broken = cont[:clen].copy()
    broken[off[victim] + 1: off[victim] + 40] = 0xFF
    rc, _, bad = cs.api.bc_decompress_host(broken, clen, out, page)
    exp_rc = chk.decompress_noheader(broken[off[victim]: off[victim + 1]].tobytes(), page)[0]
    assert exp_rc != 0 and (rc, bad) == (exp_rc, victim)
    # truncated payload and truncated index
    assert cs.api.bc_decompress_host(cont[: clen - 5].copy(), clen - 5, out, page)[0] == cs.CSNAPPY_E_DATA_MALFORMED
    assert cs.api.bc_decompress_host(cont[:1000].copy(), 1000, out, page)[0] == cs.CSNAPPY_E_DATA_MALFORMED
    assert cs.api.bc_decompress_host(cont, clen, out[: page * 10], page)[0] == cs.CSNAPPY_E_OUTPUT_INSUF


def test_batch_decompress_raw_if_full_flag(cs, chk):
    rng = np.random.default_rng(31)
    page = 4096
    raw = rng.integers(0, 256, page, dtype=np.uint8).tobytes()
    text = bytes(rng.integers(97, 100, page, dtype=np.uint8))
    streams = [raw, chk.compress_fragment(text, 13), raw[::-1], chk.compress_fragment(raw, 13)]
    expect = [raw, text, raw[::-1], raw]
    off = np.cumsum([0] + [len(s) for s in streams])  # packed back to back: arbitrary alignment
    host = np.frombuffer(b"".join(streams), dtype=np.uint8).copy()
    d_in = torch.from_numpy(host).cuda()
    d_off = torch.from_numpy(off[:-1].astype(np.int64)).cuda()
    d_len = torch.tensor([len(s) for s in streams], dtype=torch.int32).cuda()
    for lanes in (8, 16, 32, 0):
        cs.set_tuning("decompress_lanes", lanes)
        cs.set_tuning("decompress_stage_input", 0 if lanes else 4)  # last round: one lane per block
        try:
            out, out_len, status = cs.batch_decompress(d_in, d_len, len(streams), page, in_off=d_off, out_stride=page,
                                                       flags=cs.api.BATCH_RAW_IF_FULL)
            torch.cuda.synchronize()
        finally:
            cs.set_tuning("decompress_lanes", 0)
            cs.set_tuning("decompress_stage_input", 0)
        o = out.cpu().numpy()
        assert status.cpu().tolist() == [0, 0, 0, 0] and out_len.cpu().tolist() == [page] * 4
        for i, e in enumerate(expect):
            assert o[i * page:(i + 1) * page].tobytes() == e, (i, lanes)


# --------------------------------------------------------------------------- host batches + scale properties
def test_host_batch_roundtrip(cs, chk):
    pages = fuzz_pages(2024, 3000, 4096)
    B = len(pages)
    h_in = np.frombuffer(b"".join(pages), dtype=np.uint8).reshape(B, 4096)
    ostride = cs.api.out_stride_for(4096)
    h_out = np.zeros((B, ostride), dtype=np.uint8)
    h_len = np.zeros(B, dtype=np.uint32)
    cs.batch_compress_fragments_host(h_in, 4096, B, 13, h_out, h_len)
    for i in range(0, B, 37):
        assert h_out[i, : h_len[i]].tobytes() == chk.compress_fragment(pages[i], 13), i
    back = np.zeros((B, 4096), dtype=np.uint8)
    blen = np.zeros(B, dtype=np.uint32)
    st = np.ones(B, dtype=np.int32)
    cs.batch_decompress_host(h_out, ostride, h_len, B, back, 4096, 4096, blen, st)
    assert (st == 0).all() and (blen == 4096).all() and (back == h_in).all()


@pytest.mark.parametrize("bounce", [1, 0])
def test_host_paths_pinned_and_pageable_agree(cs, chk, bounce):
    """The host-buffer pipelines take pinned caller memory as it is and stage pageable memory through their own pinned
    slot buffers (copy threads; bounce=0: the round-1 behaviour, pageable memory straight into cudaMemcpyAsync):
    same bytes either way, for the strided batch calls and for the page container, over several chunks per slot."""
    pages = fuzz_pages(77, 3000, 4096) * 12  # 36000 pages: 5-6 chunks, so every pipeline slot is reused
    B = len(pages)
    flat = np.frombuffer(b"".join(pages), dtype=np.uint8)
    ostride = cs.api.out_stride_for(4096)
    cs.set_tuning("no_bounce", 0 if bounce else 1)
    try:
        res = {}
        for kind in ("pageable", "pinned"):
            mk = (lambda n, dt=torch.uint8: torch.zeros(n, dtype=dt).pin_memory()) if kind == "pinned" else \
                 (lambda n, dt=torch.uint8: torch.zeros(n, dtype=dt))
            h_in = mk(B * 4096)
            h_in.copy_(torch.from_numpy(flat.copy()))
            assert h_in.is_pinned() == (kind == "pinned")
            h_out, h_len = mk(B * ostride), mk(B, torch.int32)
            cs.batch_compress_fragments_host(h_in, 4096, B, 13, h_out, h_len)
            back, blen, st = mk(B * 4096), mk(B, torch.int32), mk(B, torch.int32)
            cs.batch_decompress_host(h_out, ostride, h_len, B, back, 4096, 4096, blen, st)
            assert int((st != 0).sum()) == 0 and int((blen != 4096).sum()) == 0 and torch.equal(back, h_in), kind
            cont = mk(cs.api.bc_max_container_length(B * 4096, 4096))
            clen = cs.api.bc_compress_host(h_in, B * 4096, cont, 13, 4096)
            back2 = mk(B * 4096)
            assert cs.api.bc_decompress_host(cont, clen, back2, 4096) == (0, B * 4096, None)
            assert torch.equal(back2, h_in), kind
            lens = h_len.numpy().astype(np.uint32)
            res[kind] = (lens.copy(), h_out.numpy().reshape(B, ostride)[np.arange(0, B, 41)].copy(), cont[:clen].numpy().copy())
        assert (res["pageable"][0] == res["pinned"][0]).all()
        for i, k in enumerate(range(0, B, 41)):
            n = res["pinned"][0][k]
            assert res["pageable"][1][i, :n].tobytes() == res["pinned"][1][i, :n].tobytes() == chk.compress_fragment(pages[k], 13), k
        assert res["pageable"][2].tobytes() == res["pinned"][2].tobytes()
    finally:
        cs.set_tuning("no_bounce", 0)


def test_packed_offsets_beyond_4_gib(cs, chk):
    """1.25 Mi mixed pages with every 5th page random: slots 5.6 GiB, PACKED payload > 4 GiB, so the u64 offsets that
    csnappy_batch_pack scans and csnappy_batch_decompress follows (in_off) cross 2^32; exact round trip + the tail pages
    (the ones whose offsets are beyond 2^32) byte-identical to the CPU reference."""
    from csnappy_b200 import synth

    B = 1310720
    d_pages = synth.mixed_pages(B, 4096, seed=0x5EED0004, device="cuda", text="urls").view(B, 4096)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(5)
    d_pages[::5] = torch.randint(0, 256, (len(range(0, B, 5)), 4096), dtype=torch.uint8, device="cuda", generator=gen)
    d_pages[1::5] = torch.randint(0, 256, (len(range(1, B, 5)), 4096), dtype=torch.uint8, device="cuda", generator=gen)
    d_pages[2::5] = torch.randint(0, 256, (len(range(2, B, 5)), 4096), dtype=torch.uint8, device="cuda", generator=gen)
    flat = d_pages.view(-1)
    ostride = cs.api.out_stride_for(4096)
    out, out_len = cs.batch_compress_fragments(flat, 4096, B, 13)
    packed, off = cs.batch_pack(out, ostride, out_len, B)
    total = int(off[-1])
    assert total > (1 << 32), total
    assert int(off[-1]) == int(out_len.to(torch.int64).sum())
    del out
    back, back_len, status = cs.batch_decompress(packed, out_len, B, 4096, in_off=off[:-1].contiguous())
    torch.cuda.synchronize()
    assert int((status != 0).sum()) == 0 and int((back_len != 4096).sum()) == 0
    assert torch.equal(back.view(B, 4096), d_pages)
    # the last pages live beyond 2^32 in the packed payload
    h_off = off[-65:].cpu().numpy()
    assert h_off[0] > (1 << 32)
    tail = packed[int(h_off[0]): int(h_off[-1])].cpu().numpy().tobytes()
    host = d_pages[B - 64:].cpu().numpy()
    exp = b"".join(chk.compress_fragment(host[i].tobytes(), 13) for i in range(64))
    assert tail == exp


def test_lane_decoder_blocks_after_failed_blocks_in_the_same_lane(cs, chk, urls):
    """Lane-per-block decoder with few lanes (one warp per SM), so every lane decodes ~10 blocks one after the other:
    a block that fails half-way leaves a line of its input in flight towards the lane's shared-memory ring; the next
    block of that lane must not see it (cp.async operations are unordered: the ring is drained before a refill)."""
    rng = np.random.default_rng(99)
    pages = [urls[o:o + 4096] for o in range(0, 4096 * 160, 4096)]
    comp = [chk.compress_fragment(p, 13) for p in pages]
    streams, caps = [], []
    for i in range(48000):
        c = bytearray(comp[i % len(comp)])
        k = int(rng.integers(0, 4))
        if k == 1:  # an invalid copy somewhere behind the first lines: offset far beyond what was produced
            at = int(rng.integers(70, len(c) - 8))
            c[at:at + 3] = bytes([0xFE, 0xFF, 0xFF])
        elif k == 2:  # output capacity too small
            pass
        streams.append(bytes(c))
        caps.append(4096 if k != 2 else int(rng.integers(100, 3000)))
    stride = (cs.csnappy_max_compressed_length(4096) + 15) // 16 * 16
    d_in, d_len, _, _ = _to_dev(streams, stride)
    d_caps = torch.tensor(caps, dtype=torch.int32).cuda()
    cs.set_tuning("decompress_stage_input", 4)
    cs.set_tuning("decompress_lane_warps", 1)
    try:
        out, out_len, status = cs.batch_decompress(d_in, d_len, len(streams), 4096, in_stride=stride, out_caps=d_caps,
                                                   out_stride=4096)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("decompress_stage_input", 0)
        cs.set_tuning("decompress_lane_warps", 0)
    st, ol, o = status.cpu().numpy(), out_len.cpu().numpy(), out.cpu().numpy().reshape(len(streams), 4096)
    memo = {}
    for i, s in enumerate(streams):
        key = (s, caps[i])
        if key not in memo:
            memo[key] = oracle.port().decompress_noheader(s, caps[i])
        rc, exp = memo[key]
        assert st[i] == rc, (i, int(st[i]), rc)
        if rc == 0:
            assert ol[i] == len(exp) and o[i, : ol[i]].tobytes() == exp, i


def test_scale_mixed_pages_roundtrip_and_oracle_sample(cs, chk):
    """256 Ki mixed 4 KiB pages (1 GiB): round trip on the device, oracle check of a sample,
    and the checksum-of-lengths property against the CPU harness on a 16 Ki page prefix."""
    from csnappy_b200 import synth

    B = 1 << 18
    d_pages = synth.mixed_pages(B, 4096, seed=0x5EED0001, device="cuda")
    out, out_len = cs.batch_compress_fragments(d_pages, 4096, B, 13)
    ostride = cs.api.out_stride_for(4096)
    back, back_len, status = cs.batch_decompress(out, out_len, B, 4096, in_stride=ostride)
    torch.cuda.synchronize()
    assert int((status != 0).sum()) == 0
    assert int((back_len != 4096).sum()) == 0
    assert torch.equal(back.view(B, 4096), d_pages.view(B, 4096))
    S = 1 << 14
    host = d_pages.view(B, 4096)[:S].cpu().numpy()
    ref_out, ref_len, _ = oracle.batch_compress(host, 13, chk.kind, threads=4)
    got_len = out_len[:S].cpu().numpy().astype(np.uint32)
    assert (got_len == ref_len).all()
    got = out.view(B, ostride)[:S].cpu().numpy()
    mask = np.arange(ostride)[None, :] < ref_len[:, None]
    assert (got[mask] == ref_out[:, :ostride][mask]).all()


def test_config3_text_fragments_32k_scale(cs, chk):
    """BASELINE config 3 shape: 32 KiB text-like fragments (wm 15 and 16), here 2048 of them (64 MiB):
    exact round trip on the device, byte identity with the reference on a sample, and the packed
    stream (size index + payload, block_compressor style) decodes again from arbitrary alignment."""
    from csnappy_b200 import synth

    n, L = 2048, 32768
    d = synth.text_fragments(n, L, device="cuda", pool_bytes=4 << 20)
    ostride = cs.api.out_stride_for(L)
    for wm in (15, 16):
        out, out_len = cs.batch_compress_fragments(d, L, n, wm)
        back, back_len, status = cs.batch_decompress(out, out_len, n, L, in_stride=ostride)
        torch.cuda.synchronize()
        assert int((status != 0).sum()) == 0 and int((back_len != L).sum()) == 0 and torch.equal(back, d)
        host = d.view(n, L)[::97].cpu().numpy()
        o = out.view(n, ostride)[::97].cpu().numpy()
        ol = out_len[::97].cpu().numpy()
        for i in range(host.shape[0]):
            assert o[i, : ol[i]].tobytes() == chk.compress_fragment(host[i].tobytes(), wm), (wm, i)
    packed, off = cs.batch_pack(out, ostride, out_len, n)
    back2, back_len2, st2 = cs.batch_decompress(packed, out_len, n, L, in_off=off[:-1].contiguous())
    torch.cuda.synchronize()
    assert int(off[-1]) == int(out_len.sum()) and int((st2 != 0).sum()) == 0 and torch.equal(back2, d)


def test_config4_decode_only_of_a_packed_corpus(cs, chk):
    """BASELINE config 4 shape: decode-only of a corpus pre-compressed BY THE REFERENCE in 4 KiB units with a
    u32 size index, payloads packed back to back (arbitrary alignment) -- checksum-of-everything style
    properties: every status 0, every length 4096, output == corpus."""
    from csnappy_b200 import synth

    n, L = 1 << 15, 4096
    corpus = synth.mixed_pages(n, L, seed=0x5EED0003, device="cpu", pool_bytes=1 << 20, text="urls").numpy().reshape(n, L)
    ref_out, ref_len, _ = oracle.batch_compress(corpus, 13, chk.kind, threads=8)
    offs = np.concatenate([[0], np.cumsum(ref_len.astype(np.int64))])
    packed = np.zeros(int(offs[-1]) + 16, dtype=np.uint8)
    mask = np.arange(ref_out.shape[1])[None, :] < ref_len[:, None]
    packed[: int(offs[-1])] = ref_out[mask]
    out, out_len, status = cs.batch_decompress(torch.from_numpy(packed).cuda(),
                                               torch.from_numpy(ref_len.astype(np.int32)).cuda(), n, L,
                                               in_off=torch.from_numpy(offs[:-1].copy()).cuda(), out_stride=L)
    torch.cuda.synchronize()
    assert int((status != 0).sum()) == 0 and int((out_len != L).sum()) == 0
    assert (out.cpu().numpy().reshape(n, L) == corpus).all()


# --------------------------------------------------------------------------- round 2 additions to the boundary
def test_batch_compress_whole_buffers_with_header(cs, chk, urls):
    """csnappy_batch_compress: many WHOLE buffers per call, each framed like csnappy_compress
    (csnappy_compress.c:621-656) -- byte-identical to the reference per buffer, at several table sizes."""
    rng = np.random.default_rng(41)
    text = bytes(rng.integers(97, 102, 120000, dtype=np.uint8))
    bufs = [b"", b"a", text[:14], text[:15], text[:100], text[:32767], text[:32768], text[:32769], text[:70001],
            urls[:100000], bytes(50000), rng.integers(0, 256, 40000, dtype=np.uint8).tobytes(), urls]
    offs, pos = [], 0
    for b in bufs:
        offs.append(pos)
        pos += len(b) + 3  # arbitrary alignment of every buffer
    host = np.zeros(pos + 16, dtype=np.uint8)
    for o, b in zip(offs, bufs):
        host[o:o + len(b)] = np.frombuffer(b, dtype=np.uint8)
    d_in = torch.from_numpy(host).cuda()
    for wm in (9, 13, 15, 16):
        out, out_len, stride = cs.api.batch_compress(d_in, offs, [len(b) for b in bufs], wm)
        o, ol = out.cpu().numpy(), out_len.cpu().numpy()
        for i, b in enumerate(bufs):
            assert o[i * stride: i * stride + ol[i]].tobytes() == chk.compress(b, wm), (i, len(b), wm)


def test_bc_container_multi_device_entry_points(cs, chk, urls):
    """csnappy_bc_*_host_multi from ONE process: all visible devices, and device 0 listed three times (three workers and
    contexts exercise the chunk-position hand-over on a single GPU).  Bytes identical to the single-device writer."""
    from csnappy_b200 import synth

    B, page = 30000, 4096
    h_in = synth.mixed_pages(B, page, seed=78, device="cuda", pool_bytes=1 << 20).cpu().numpy()
    cap = cs.api.bc_max_container_length(B * page, page)
    ref = np.zeros(cap, dtype=np.uint8)
    clen = cs.api.bc_compress_host(h_in, B * page, ref, 13, page)
    for devices in (None, [0, 0, 0]):
        cont = np.zeros(cap, dtype=np.uint8)
        assert cs.api.bc_compress_host_multi(h_in, B * page, cont, 13, page, devices=devices) == clen
        assert (cont[:clen] == ref[:clen]).all()
        out = np.zeros(B * page, dtype=np.uint8)
        assert cs.api.bc_decompress_host_multi(cont, clen, out, page, devices=devices) == (0, B * page, None)
        assert (out == h_in).all()
    # a corrupted page is reported by index through the multi-device reader too
    idx = ref[4:4 + 4 * B].view(np.uint32)
    off = 4 + 4 * B + np.concatenate([[0], np.cumsum(idx.astype(np.int64))])
    victim = next(i for i in range(17000, B) if 100 < idx[i] < page)
    broken = ref[:clen].copy()
    broken[off[victim] + 1: off[victim] + 40] = 0xFF
    out = np.zeros(B * page, dtype=np.uint8)
    rc, _, bad = cs.api.bc_decompress_host_multi(broken, clen, out, page, devices=[0, 0])
    assert rc == chk.decompress_noheader(broken[off[victim]: off[victim + 1]].tobytes(), page)[0] != 0 and bad == victim


def test_dropin_large_buffer_pipeline_and_concurrent_callers(cs, chk, urls):
    """csnappy_compress of a multi-chunk buffer goes through the chunk pipeline; concurrent callers on disjoint buffers
    (the reference is re-entrant, csnappy.h:46-72) each get their own staging context and the same bytes."""
    import threading

    big = (urls * 14)[: 9 * 1024 * 1024 + 12345]  # > 8 MiB: several pipeline chunks
    c = cs.csnappy_compress(big, 15)
    assert c == chk.compress(big, 15)
    assert cs.csnappy_decompress(c, len(big)) == (0, big)
    inputs = [urls[i * 1000: i * 1000 + 150000 + 777 * i] for i in range(8)]
    want = [chk.compress(x, 16) for x in inputs]
    got = [None] * len(inputs)
    back = [None] * len(inputs)

    def work(i):
        for _ in range(3):
            got[i] = cs.csnappy_compress(inputs[i], 16)
            back[i] = cs.csnappy_decompress(got[i], len(inputs[i]))
            page = cs.csnappy_compress_fragment(inputs[i][:4096], 13)
            assert page == chk.compress_fragment(inputs[i][:4096], 13)

    th = [threading.Thread(target=work, args=(i,)) for i in range(len(inputs))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert got == want
    assert back == [(0, x) for x in inputs]


@pytest.mark.parametrize("stream_min", [0, -1])
def test_single_long_streams_parallel_decoder_vs_oracle(cs, chk, urls, urls_snappy, baddata3, unaligned_pair, stream_min):
    """f-4: ONE long stream through the drop-in csnappy_decompress_noheader / csnappy_decompress -- the parallel
    stream decoder (stream_kernel.cu; stream_min 0) and the serial warp-per-stream path (-1) against the oracle:
    fixtures, multi-fragment streams of every entropy class, corrupted / truncated / extended / under-sized."""
    uu_s, uu_b = unaligned_pair
    rng = np.random.default_rng(77)
    cs.set_tuning("stream_decode_min", stream_min)
    try:
        rc, out = cs.csnappy_decompress(urls_snappy, len(urls))
        assert rc == 0 and out == urls
        assert cs.csnappy_decompress(baddata3, 130378)[0] == -5
        rc, out = cs.csnappy_decompress(uu_s, len(uu_b))
        assert rc == 0 and out == uu_b
        assert cs.csnappy_decompress(urls_snappy, len(urls) - 1)[0] == cs.CSNAPPY_E_OUTPUT_INSUF
        bodies = []
        for k, page in enumerate(fuzz_pages(606, 14, 90000 + 7777)):
            data = page + urls[k * 5000: k * 5000 + 70000] + bytes(3000 * (k % 3)) + page[:20000]
            bodies.append((data, chk.compress(data, 15 if k % 2 else 16)))
        cases = []
        for k, (data, comp) in enumerate(bodies):
            hlen, n = chk.get_uncompressed_length(comp)
            raw = comp[hlen:]
            cases.append((raw, n))  # valid
            cases.append((raw, n - 1 - int(rng.integers(0, n // 2))))  # under-sized: -3 somewhere
            d = bytearray(raw)
            for _ in range(1 + k % 3):
                d[int(rng.integers(0, len(d)))] ^= int(rng.integers(1, 256))
            cases.append((bytes(d), n))  # flipped bytes
            cases.append((raw[: int(rng.integers(len(raw) // 2, len(raw)))], n))  # truncated
            cases.append((raw + bytes(rng.integers(0, 256, 5, dtype=np.uint8)), n + 300))  # extended
        n_err = 0
        for i, (s, cap) in enumerate(cases):
            rc, exp = oracle.port().decompress_noheader(s, cap)
            got_rc, got = cs.csnappy_decompress_noheader(s, cap)
            assert got_rc == rc, (i, stream_min, len(s), cap)
            if rc == 0:
                assert got == exp, (i, stream_min)
            else:
                n_err += 1
        assert n_err >= len(cases) // 3
    finally:
        cs.set_tuning("stream_decode_min", 0)
