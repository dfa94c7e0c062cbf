#!/usr/bin/env python
"""Long randomized parity run on the GPU box: many seeds / block sizes / table sizes / lane groups,
compressed bytes and decoder results compared with the unmodified reference (oracle/_ref).  The compress leg
also gets blocks built to drive the parse through the kernel's rare paths (tests/compress_cases.py: hash-slot
sharing in stride-1 and strided windows, in-window copies, the scan end, length and offset boundaries); the decode
leg gets random streams of every tag form (tests/streams.py), which the compressor never writes.  The container leg
writes a page container of random page size and length, corrupts its index and payload at random and compares the
reader with the restated reader (tests/containers.py), through the host call, the device-buffer reader and a random
batch of device page reads.  The framed leg round-trips a random buffer through the framing
format, compares the stream with the restated writer, corrupts it at random and compares the reader with the restated
reader (tests/framed.py).  The batched-framed leg writes several random buffers in one csnappy_framed_batch_compress
call, corrupts some of the streams, and reads valid and hostile streams together in one csnappy_framed_batch_decompress
call, each against the restated writer and reader.

    python tools/fuzz_gpu.py [seconds] [seed]
"""
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
sys.path.insert(0, "tests")
import csnappy_b200 as cs
import oracle
import compress_cases
import containers
import framed
from cases import fuzz_pages
from streams import random_stream
from test_gpu_bc_device import restated_index, restated_request

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 120.0
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 20261017
chk = oracle.best()
rng = np.random.default_rng(seed)
t0 = time.time()
rounds = blocks = streams = pages_read = pages_requested = framed_streams = batch_framed = 0
while time.time() - t0 < budget:
    size = int(rng.choice([17, 64, 300, 1000, 4096, 4096, 4096, 5000, 16384, 32768]))
    wm = int(rng.integers(9, 17))
    lanes = int(rng.choice([8, 16, 32]))
    count = int(rng.integers(20, 120))
    pages = fuzz_pages(int(rng.integers(1 << 30)), count, size)
    if size >= 1000:  # a few constructed blocks per round (building one takes 0.1-1 s)
        themes = ("share", "strided", "emit", "share")
        for i in rng.choice(count, min(count, 3), replace=False):
            try:
                c = compress_cases.build_block(int(rng.integers(1 << 30)), size, wm, themes[int(i) % 4])
            except compress_cases.Plan:
                c = None
            if c is not None:
                pages[int(i)] = c.data
    # ragged lengths
    lens = np.array([int(rng.integers(0, size + 1)) if rng.random() < 0.3 else size for _ in pages], dtype=np.int32)
    host = np.zeros((count, size), dtype=np.uint8)
    for i, p in enumerate(pages):
        host[i] = np.frombuffer(p, dtype=np.uint8)
    cs.set_tuning("compress_lanes", lanes)
    cs.set_tuning("decompress_lanes", lanes)
    cs.set_tuning("compress_stage_input", int(rng.choice([0, 1, 2])) if lanes == 32 else 0)  # staged / read from global
    cs.set_tuning("decompress_stage_input", int(rng.choice([0, 0, 1, 3, 4])))  # default routing / staged / global / lane
    d_in, d_len = torch.from_numpy(host).cuda(), torch.from_numpy(lens).cuda()
    out, out_len = cs.batch_compress_fragments(d_in, size, count, wm, in_len=d_len)
    torch.cuda.synchronize()
    ostride = cs.api.out_stride_for(size)
    o = out.cpu().numpy().reshape(-1)[: count * ostride].reshape(count, ostride)
    ol = out_len.cpu().numpy()
    comp = []
    for i in range(count):
        ref = chk.compress_fragment(pages[i][: lens[i]], wm)
        got = o[i, : ol[i]].tobytes()
        assert got == ref, ("compress", size, wm, lanes, i, int(lens[i]))
        comp.append(ref)
    blocks += count
    # decode: valid, corrupted and truncated streams, capacity sometimes too small
    strs, caps = [], []
    for i, c in enumerate(comp):
        d = bytearray(c)
        k = int(rng.integers(0, 6))
        if k == 1 and len(d) > 2:
            for _ in range(int(rng.integers(1, 4))):
                d[int(rng.integers(0, len(d)))] = int(rng.integers(0, 256))
        elif k == 2 and len(d) > 2:
            d = d[: int(rng.integers(1, len(d)))]
        elif k == 3:
            d += bytes(rng.integers(0, 256, int(rng.integers(1, 9)), dtype=np.uint8))
        strs.append(bytes(d))
        caps.append(int(lens[i]) if k != 4 else int(rng.integers(0, max(1, int(lens[i])))))
    stride = (cs.csnappy_max_compressed_length(size) + 16 + 15) // 16 * 16
    for _ in range(int(rng.integers(1, count // 4 + 2))):
        s = random_stream(int(rng.integers(1 << 30)), int(rng.integers(1, size + 1)))
        if len(s.buf) <= stride:  # capacity at most the block size: sometimes short of the stream's output
            strs.append(bytes(s.buf))
            caps.append(min(s.produced, size))
    n_dec = len(strs)
    hs = np.zeros((n_dec, stride), dtype=np.uint8)
    sl = np.zeros(n_dec, dtype=np.int32)
    for i, s in enumerate(strs):
        hs[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
        sl[i] = len(s)
    ocap = (size + 15) // 16 * 16
    res = cs.batch_decompress(torch.from_numpy(hs).cuda(), torch.from_numpy(sl).cuda(), n_dec, size, in_stride=stride,
                              out_caps=torch.tensor(caps, dtype=torch.int32).cuda(), out_stride=max(ocap, 16))
    torch.cuda.synchronize()
    bo, bl, st = (x.cpu().numpy() for x in res)
    for i, s in enumerate(strs):
        rc, exp = oracle.port().decompress_noheader(s, caps[i])  # the port defines the truncated-tag case as -5
        assert st[i] == rc, ("status", size, wm, lanes, i, int(st[i]), rc, s.hex()[:60])
        if rc == 0:
            assert bl[i] == len(exp) and bo[i * max(ocap, 16): i * max(ocap, 16) + bl[i]].tobytes() == exp, ("bytes", size, lanes, i)
    streams += n_dec
    # container: random page size and length, the index and payloads corrupted at random, against the restated reader
    page = int(rng.choice([1, 17, 1000, 4095, 4096, 4097, 20000, 32768]))
    data = containers.mixed_bytes(int(rng.integers(1 << 30)), int(rng.integers(1, 600 * page + 2)), scale=max(page, 64))
    cont = np.zeros(cs.api.bc_max_container_length(len(data), page), dtype=np.uint8)
    clen = cs.api.bc_compress_host(np.frombuffer(data, dtype=np.uint8), len(data), cont, wm, page)
    assert cont[:clen].tobytes() == containers.ref_container(chk, data, page, wm), ("container", page, len(data), wm)
    broken = bytearray(cont[:clen].tobytes())
    nr = (len(data) + page - 1) // page
    for _ in range(int(rng.integers(0, 4))):
        i = int(rng.integers(0, nr))
        broken[4 + 4 * i: 8 + 4 * i] = int(rng.choice([0, page - 1, page, page + 1, 32 + page + page // 6 + 1,
                                                        int(rng.integers(0, 2 * page + 40))])).to_bytes(4, "little")
    for _ in range(int(rng.integers(0, 4))):
        broken[int(rng.integers(4 + 4 * nr, len(broken) + 1)) - 1] ^= int(rng.integers(1, 256))
    if rng.random() < 0.2:
        broken = broken[: int(rng.integers(4, len(broken) + 1))]
    want = containers.read_container(bytes(broken), page, nr * page)
    out = np.zeros(nr * page, dtype=np.uint8)
    rc, olen, bad = cs.api.bc_decompress_host(np.frombuffer(bytes(broken), dtype=np.uint8), len(broken), out, page)
    assert (rc, olen, bad) == want.key(), ("container read", page, len(data), want.key(), (rc, olen, bad))
    for i, b in want.pages.items():
        assert out[i * page: i * page + len(b)].tobytes() == b, ("container page", page, i)
    # the same broken container in device memory: the whole-container reader, then a random batch of page reads
    d_b = torch.frombuffer(bytearray(broken), dtype=torch.uint8).cuda()
    d_out, res = cs.api.bc_decompress_device(d_b, len(broken), page, nr * page)
    torch.cuda.synchronize()
    r = res.cpu().tolist()
    assert (r[1], r[0], None if r[2] == -1 else r[2]) == want.key(), ("device container read", page, want.key(), r)
    out = d_out.cpu().numpy()
    for i, b in want.pages.items():
        assert out[i * page: i * page + len(b)].tobytes() == b, ("device container page", page, i)
    rc, idx, n_idx = cs.api.bc_index_device(d_b, len(broken), page)
    assert rc == (containers.E_DATA_MALFORMED if len(broken) < 4 + 4 * nr else 0), ("index", rc)
    if rc == 0:
        offs = restated_index(bytes(broken), page)[1]
        assert [int(x) & (2**64 - 1) for x in idx[:n_idx].cpu().tolist()] == offs, ("index", page)
        req = rng.integers(0, nr + 2, int(rng.integers(1, 200))).astype(np.uint32)
        stride = page + int(rng.choice([0, 0, 5, 16]))
        o, ol, st = cs.api.bc_decompress_pages_device(d_b, idx, n_idx, torch.from_numpy(req.view(np.int32)).cuda(), page,
                                                      len(broken), out_stride=stride)
        torch.cuda.synchronize()
        o, ol, st = o.cpu().numpy(), ol.cpu().tolist(), st.cpu().tolist()
        for k, p in enumerate(req.tolist()):
            rc_k, b = restated_request(bytes(broken), page, offs, p, nr)
            assert (st[k], ol[k]) == (rc_k, len(b) if b is not None else 0), ("page read", page, p, st[k], rc_k)
            if b is not None:
                assert o[k * stride:k * stride + len(b)].tobytes() == b, ("page read bytes", page, p)
        pages_requested += len(req)
    pages_read += nr
    # framed: a random buffer round-trips and its stream equals the restated writer; random corruptions of it give the
    # restated reader's (rc, out_length, failed_offset) and valid prefix
    data = containers.mixed_bytes(int(rng.integers(1 << 30)), int(rng.integers(0, 5 * framed.CHUNK)), scale=int(rng.integers(64, 70000)))
    s = cs.api.framed_compress(data, wm)
    assert s == framed.write_framed(data, wm), ("framed write", len(data), wm)
    assert cs.api.framed_decompress(s, len(data)) == (0, data, None), ("framed round trip", len(data))
    broken = bytearray(s)
    for _ in range(int(rng.integers(1, 4))):
        broken[int(rng.integers(0, len(broken)))] ^= 1 << int(rng.integers(0, 8))
    if rng.random() < 0.2:
        broken = broken[: int(rng.integers(0, len(broken) + 1))]
    cap = len(data) - int(rng.integers(0, 2)) * int(rng.integers(0, len(data) + 1))
    want = framed.read_framed(bytes(broken), cap)
    rc, out, bad = cs.api.framed_decompress(bytes(broken), cap)
    assert (rc, len(out), bad) == want.key() and out == want.data, ("framed read", len(data), want.key(), (rc, len(out), bad))
    framed_streams += 1
    # batched framed: valid and hostile streams mixed in one call, every one against the restatement
    bufs = [containers.mixed_bytes(int(rng.integers(1 << 30)), int(rng.choice([0, int(rng.integers(0, 300)),
                                                                               int(rng.integers(0, 3 * framed.CHUNK))])),
                                   scale=int(rng.integers(64, 70000))) for _ in range(int(rng.integers(1, 12)))]
    zs = cs.api.framed_batch_compress(bufs, wm)
    assert zs == [framed.write_framed(b, wm) for b in bufs], ("framed batch write", wm, [len(b) for b in bufs])
    hostile, caps = [], []
    for z, b in zip(zs, bufs):
        z = bytearray(z)
        if rng.random() < 0.5 and z:
            for _ in range(int(rng.integers(1, 4))):
                z[int(rng.integers(0, len(z)))] ^= 1 << int(rng.integers(0, 8))
        if rng.random() < 0.2:
            z = z[: int(rng.integers(0, len(z) + 1))]
        hostile.append(bytes(z))
        caps.append(len(b) - int(rng.integers(0, 2)) * int(rng.integers(0, len(b) + 1)))
    got = cs.api.framed_batch_decompress(hostile, caps)
    for z, c, g in zip(hostile, caps, got):
        want = framed.read_framed(z, c)
        assert (g[0], len(g[1]), g[2]) == want.key() and g[1] == want.data, ("framed batch read", want.key(), g[0], len(g[1]), g[2])
    batch_framed += len(bufs)
    rounds += 1
cs.set_tuning("compress_lanes", 0)
cs.set_tuning("decompress_lanes", 0)
cs.set_tuning("compress_stage_input", 0)
cs.set_tuning("decompress_stage_input", 0)
print(f"fuzz ok: {rounds} rounds, {blocks} blocks compressed byte-identically, {streams} streams decoded with identical results, "
      f"{pages_read} container pages written and read as restated, {pages_requested} device page reads as restated, "
      f"{framed_streams} framed streams written, corrupted and read as restated, "
      f"{batch_framed} streams through the batched framed calls in {time.time() - t0:.0f} s")
