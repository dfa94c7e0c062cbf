#!/usr/bin/env python
"""Long randomized parity run on the GPU box: many seeds / block sizes / table sizes / lane groups,
compressed bytes and decoder results compared with the unmodified reference (oracle/_ref).  The compress leg
also gets blocks built to drive the parse through the kernel's rare paths (tests/compress_cases.py: hash-slot
sharing in stride-1 and strided windows, in-window copies, the scan end, length and offset boundaries); the decode
leg gets random streams of every tag form (tests/streams.py), which the compressor never writes.

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
from cases import fuzz_pages
from streams import random_stream

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 120.0
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 20261017
chk = oracle.best()
rng = np.random.default_rng(seed)
t0 = time.time()
rounds = blocks = streams = 0
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
    rounds += 1
cs.set_tuning("compress_lanes", 0)
cs.set_tuning("decompress_lanes", 0)
cs.set_tuning("compress_stage_input", 0)
cs.set_tuning("decompress_stage_input", 0)
print(f"fuzz ok: {rounds} rounds, {blocks} blocks compressed byte-identically, {streams} streams decoded with identical results "
      f"in {time.time() - t0:.0f} s")
