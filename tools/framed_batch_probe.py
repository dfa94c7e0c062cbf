"""Throughput of the batched framing calls on one GPU, device resident: many streams of one size written and read in
one call, against the same streams through a loop of single framed calls (a timed subset spread over the input), and
against csnappy_batch_compress / csnappy_batch_decompress(WITH_HEADER) over the same buffers (the unframed ceiling).
The declared-length call is timed too.

    python tools/framed_batch_probe.py [--gib 4] [--passes 3] [--sizes 4096,65536,1048576] [--out profiles/framed_batch_probe.json]

Inputs are larger than L2 (4 GiB by default): text (32 MiB word-stream pool, 64 KiB windows at seeded offsets) and
mixed (zram-style 4 KiB pages: text / zero / random), cut into streams of each size.  Every leg is warmed up once,
then timed over --passes with CUDA events; GB/s are of uncompressed bytes.  The card's name and power limit are read
in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from csnappy_b200 import api, synth  # noqa: E402
from csnappy_b200._lib import lib  # noqa: E402
from tools.framed_probe import card, gbs, timed  # noqa: E402

SINGLE_BYTES = 64 << 20  # uncompressed bytes of the single-call subset


def leg(d, size, passes):
    L = lib()
    s = torch.cuda.current_stream().cuda_stream
    n = d.numel() // size * size
    k = n // size
    offs = np.ascontiguousarray(np.arange(k, dtype=np.uint64) * np.uint64(size))
    lens = np.full(k, size, dtype=np.uint64)
    m = L.csnappy_framed_max_length(size)
    out_off = np.ascontiguousarray(np.arange(k, dtype=np.uint64) * np.uint64(m))
    res = {"streams": k, "bytes": n}
    out = torch.empty(k * m, dtype=torch.uint8, device="cuda")
    olen = torch.empty(k, dtype=torch.int64, device="cuda")
    ws_n = L.csnappy_framed_batch_compress_workspace(lens.ctypes.data, k)
    ws = torch.empty(ws_n, dtype=torch.uint8, device="cuda")

    def comp():
        assert L.csnappy_framed_batch_compress(d.data_ptr(), offs.ctypes.data, lens.ctypes.data, k, out.data_ptr(),
                                               out_off.ctypes.data, out.numel(), olen.data_ptr(), 16, ws.data_ptr(), ws_n,
                                               s) == 0

    res["framed_batch_compress_gbs"] = gbs(n, timed(comp, passes))
    del ws
    torch.cuda.empty_cache()
    zl = np.ascontiguousarray(olen.cpu().numpy().astype(np.uint64))
    res["framed_ratio"] = round(float(zl.sum()) / n, 4)
    length = torch.empty(k, dtype=torch.int64, device="cuda")
    st = torch.empty(k, dtype=torch.int32, device="cuda")
    res["decompressed_length_gbs"] = gbs(n, timed(lambda: L.csnappy_framed_batch_decompressed_length(
        out.data_ptr(), out_off.ctypes.data, zl.ctypes.data, k, length.data_ptr(), st.data_ptr(), s), passes))
    assert bool((length == size).all()) and bool((st == 0).all())
    dst = torch.empty(n, dtype=torch.uint8, device="cuda")
    fo = torch.empty(k, dtype=torch.int64, device="cuda")
    wsd_n = L.csnappy_framed_batch_decompress_workspace(zl.ctypes.data, k)
    wsd = torch.empty(wsd_n, dtype=torch.uint8, device="cuda")

    def dec():
        assert L.csnappy_framed_batch_decompress(out.data_ptr(), out_off.ctypes.data, zl.ctypes.data, k, dst.data_ptr(),
                                                 offs.ctypes.data, lens.ctypes.data, length.data_ptr(), st.data_ptr(),
                                                 fo.data_ptr(), wsd.data_ptr(), wsd_n, s) == 0

    res["framed_batch_decompress_gbs"] = gbs(n, timed(dec, passes))
    assert bool((st == 0).all()) and bool((length == size).all()) and torch.equal(dst, d[:n])
    del wsd
    torch.cuda.empty_cache()
    # single calls on a subset spread over the whole input
    sub = max(1, min(k, SINGLE_BYTES // size))
    pick = np.linspace(0, k - 1, sub).astype(np.int64)
    one_ws = torch.empty(max(L.csnappy_framed_compress_workspace(size), L.csnappy_framed_decompress_workspace(m)),
                         dtype=torch.uint8, device="cuda")
    sout = torch.empty(m, dtype=torch.uint8, device="cuda")
    r = torch.empty(4, dtype=torch.int64, device="cuda")

    def scomp():
        for i in pick:
            assert L.csnappy_framed_compress(d.data_ptr() + int(i) * size, size, sout.data_ptr(), m, r.data_ptr(), 16,
                                             one_ws.data_ptr(), one_ws.numel(), s) == 0

    def sdec():
        for i in pick:
            assert L.csnappy_framed_decompress(out.data_ptr() + int(out_off[i]), int(zl[i]), dst.data_ptr() + int(i) * size,
                                               size, r.data_ptr(), r.data_ptr() + 8, r.data_ptr() + 16, one_ws.data_ptr(),
                                               one_ws.numel(), s) == 0

    res["single_calls_streams_timed"] = int(sub)
    res["single_compress_loop_gbs"] = gbs(sub * size, timed(scomp, passes))
    res["single_decompress_loop_gbs"] = gbs(sub * size, timed(sdec, passes))
    del one_ws, out
    torch.cuda.empty_cache()
    # the unframed ceiling: csnappy_batch_compress / csnappy_batch_decompress(WITH_HEADER) of the same buffers
    len32 = np.full(k, size, dtype=np.uint32)
    stride = (5 + size + size // 6 + 32 * max(1, -(-size // 32768)) + 15) // 16 * 16
    bout = torch.empty(k * stride, dtype=torch.uint8, device="cuda")
    blen = torch.empty(k, dtype=torch.int32, device="cuda")
    wsb_n = L.csnappy_batch_compress_workspace(len32.ctypes.data, 0, k)
    wsb = torch.empty(wsb_n, dtype=torch.uint8, device="cuda")

    def bcomp():
        assert L.csnappy_batch_compress(d.data_ptr(), offs.ctypes.data, 0, len32.ctypes.data, 0, k, bout.data_ptr(), stride,
                                        blen.data_ptr(), 16, wsb.data_ptr(), wsb_n, s) == 0

    res["batch_compress_gbs"] = gbs(n, timed(bcomp, passes))
    del wsb
    torch.cuda.empty_cache()
    ol = torch.empty(k, dtype=torch.int32, device="cuda")

    def bdec():
        assert L.csnappy_batch_decompress(bout.data_ptr(), None, stride, blen.data_ptr(), k, dst.data_ptr(), size, None,
                                          size, ol.data_ptr(), st.data_ptr(), api.BATCH_WITH_HEADER, s) == 0

    res["batch_decompress_with_header_gbs"] = gbs(n, timed(bdec, passes))
    assert torch.equal(dst, d[:n])
    del bout, dst
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--sizes", default="4096,65536,1048576")
    ap.add_argument("--out", default="profiles/framed_batch_probe.json")
    a = ap.parse_args()
    sizes = [int(x) for x in a.sizes.split(",")]
    n = int(a.gib * (1 << 30)) // max(sizes) * max(sizes)
    rep = {"card": card(), "bytes": n, "passes": a.passes, "single_call_subset_bytes": SINGLE_BYTES, "classes": {}}
    for cls in ("text", "mixed"):
        d = synth.text_fragments(n // 65536, 65536) if cls == "text" else synth.mixed_pages(n // 4096, 4096)
        rep["classes"][cls] = {}
        for size in sizes:
            rep["classes"][cls][str(size)] = leg(d, size, a.passes)
            print(cls, size, json.dumps(rep["classes"][cls][str(size)]), flush=True)
        del d
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps(rep))


if __name__ == "__main__":
    main()
