"""Throughput of the page container calls on device buffers, on one GPU, against the raw batch calls on the same pages.

    python tools/bc_device_probe.py [--pages 1048576] [--passes 3] [--out profiles/bc_device_probe.json]

Workload: bench.py's, 1 Mi zram-style mixed 4 KiB pages (csnappy_b200/synth.py: text / zero / random), wm 13, all in
device memory (4 GiB of pages, larger than L2).  Legs, each pair warmed up and then timed alternately over --passes
with CUDA events:
  1. csnappy_bc_compress (container) vs csnappy_batch_compress_fragments (strided slots) of the same pages;
  2. csnappy_bc_decompress of that container vs csnappy_batch_decompress of the same fragments in strided slots;
  3. csnappy_bc_index alone at 1 Mi and 16 Mi entries vs csnappy_batch_pack with d_packed = NULL (the single-CTA
     scan_kernel) over the same sizes;
  4. csnappy_bc_decompress_pages of 1 Ki, 64 Ki and 1 Mi random page numbers of the container.
GB/s are of uncompressed page bytes (produced bytes for the page reads).  The card's name and power limit are read in
the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from csnappy_b200 import synth  # noqa: E402
from csnappy_b200._lib import lib  # noqa: E402
from tools.framed_probe import card, gbs  # noqa: E402

PAGE, WM = 4096, 13


def pair(fa, fb, passes):
    """Warm both, then time them alternately; -> (seconds per call of a, of b)."""
    fa(), fb()
    torch.cuda.synchronize()
    ta = tb = 0.0
    for _ in range(passes):
        for f, which in ((fa, 0), (fb, 1)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            torch.cuda.synchronize()
            if which == 0:
                ta += a.elapsed_time(b) / 1e3
            else:
                tb += a.elapsed_time(b) / 1e3
    return ta / passes, tb / passes


def one(f, passes):
    return pair(f, lambda: None, passes)[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pages", type=int, default=1 << 20)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--out", default="profiles/bc_device_probe.json")
    args = ap.parse_args()
    L = lib()
    s = torch.cuda.current_stream().cuda_stream
    B = args.pages
    n = B * PAGE
    res = {"card": card(), "pages": B, "page_size": PAGE, "wm": WM, "passes": args.passes,
           "workload": "synth.mixed_pages (bench.py's mixed 4 KiB pages), device resident"}
    d = synth.mixed_pages(B, PAGE)
    # 1. writer vs raw fragments
    cap = L.csnappy_bc_max_container_length(n, PAGE)
    cont = torch.empty(cap, dtype=torch.uint8, device="cuda")
    clen = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws_n = L.csnappy_bc_compress_workspace(n, PAGE)
    ws = torch.empty(ws_n, dtype=torch.uint8, device="cuda")
    stride = (32 + PAGE + PAGE // 6 + 15) // 16 * 16
    frag = torch.empty(B * stride, dtype=torch.uint8, device="cuda")
    flen = torch.empty(B, dtype=torch.int32, device="cuda")

    def write():
        assert L.csnappy_bc_compress(d.data_ptr(), n, PAGE, cont.data_ptr(), cap, clen.data_ptr(), WM, ws.data_ptr(),
                                     ws_n, s) == 0

    def frags():
        assert L.csnappy_batch_compress_fragments(d.data_ptr(), None, PAGE, None, PAGE, B, frag.data_ptr(), stride,
                                                  flen.data_ptr(), WM, 0, s) == 0

    tw, tf = pair(write, frags, args.passes)
    clen_v = int(clen.item())
    res["write"] = {"bc_compress_gbs": gbs(n, tw), "batch_compress_fragments_gbs": gbs(n, tf),
                    "bc_compress_ms": round(tw * 1e3, 3), "batch_compress_fragments_ms": round(tf * 1e3, 3),
                    "container_ratio": round(clen_v / n, 4)}
    del ws
    torch.cuda.empty_cache()
    # 2. whole read vs raw batch decode of the fragments
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    olen = torch.zeros(1, dtype=torch.int64, device="cuda")
    words = torch.full((2,), -1, dtype=torch.int32, device="cuda")
    wsd_n = L.csnappy_bc_decompress_workspace(clen_v, PAGE, n)
    wsd = torch.empty(wsd_n, dtype=torch.uint8, device="cuda")
    rout = torch.empty(n, dtype=torch.uint8, device="cuda")
    rlen = torch.empty(B, dtype=torch.int32, device="cuda")
    rst = torch.empty(B, dtype=torch.int32, device="cuda")

    def read():
        assert L.csnappy_bc_decompress(cont.data_ptr(), clen_v, PAGE, out.data_ptr(), n, olen.data_ptr(),
                                       words.data_ptr(), words.data_ptr() + 4, wsd.data_ptr(), wsd_n, s) == 0

    def raw_read():
        assert L.csnappy_batch_decompress(frag.data_ptr(), None, stride, flen.data_ptr(), B, rout.data_ptr(), PAGE, None,
                                          PAGE, rlen.data_ptr(), rst.data_ptr(), 0, s) == 0

    tr, trr = pair(read, raw_read, args.passes)
    assert int(words[0].item()) == 0 and int(olen.item()) == n and torch.equal(out, d)
    assert bool((rst == 0).all()) and torch.equal(rout, d)
    res["read"] = {"bc_decompress_gbs": gbs(n, tr), "batch_decompress_gbs": gbs(n, trr),
                   "bc_decompress_ms": round(tr * 1e3, 3), "batch_decompress_ms": round(trr * 1e3, 3)}
    del rout, rlen, rst, wsd
    torch.cuda.empty_cache()
    # 3. the index scan alone vs the single-CTA scan_kernel, 1 Mi and 16 Mi entries
    entries = cont[4:4 + 4 * B].view(torch.int32).clone()
    res["index"] = {}
    for mult in (1, 16):
        m = B * mult
        lens = entries.repeat(mult)
        buf = torch.empty(4 + 4 * m, dtype=torch.uint8, device="cuda")
        buf[:4] = torch.tensor([m], dtype=torch.int32).view(torch.uint8).cuda()
        buf[4:] = lens.view(torch.uint8)
        length = 4 + 4 * m + int(lens.to(torch.int64).sum().item())  # the payloads are not read by the index call
        idx = torch.empty(m, dtype=torch.int64, device="cuda")
        off = torch.empty(m + 1, dtype=torch.int64, device="cuda")
        nr = C.c_uint32(0)

        def index():
            assert L.csnappy_bc_index(buf.data_ptr(), length, PAGE, idx.data_ptr(), m, C.byref(nr), s) == 0

        def scan():
            assert L.csnappy_batch_pack(None, 0, lens.data_ptr(), m, None, off.data_ptr(), s) == 0

        ti, ts = pair(index, scan, args.passes)
        assert torch.equal(idx, off[:m] + 4 + 4 * m)
        res["index"][f"{m}_entries"] = {"bc_index_us": round(ti * 1e6, 1), "scan_kernel_us": round(ts * 1e6, 1)}
        del buf, idx, off, lens
        torch.cuda.empty_cache()
    # 4. random page reads from the 1 Mi-page container
    idx = torch.empty(B, dtype=torch.int64, device="cuda")
    nr = C.c_uint32(0)
    assert L.csnappy_bc_index(cont.data_ptr(), clen_v, PAGE, idx.data_ptr(), B, C.byref(nr), s) == 0
    res["page_reads"] = {}
    for k in (1 << 10, 1 << 16, 1 << 20):
        pages = torch.from_numpy(np.random.default_rng(k).integers(0, B, k).astype(np.int32)).cuda()
        po = torch.empty(k * PAGE, dtype=torch.uint8, device="cuda")
        pl = torch.empty(k, dtype=torch.int32, device="cuda")
        ps = torch.empty(k, dtype=torch.int32, device="cuda")
        wsp_n = L.csnappy_bc_decompress_pages_workspace(k)
        wsp = torch.empty(wsp_n, dtype=torch.uint8, device="cuda")

        def reads():
            assert L.csnappy_bc_decompress_pages(cont.data_ptr(), clen_v, PAGE, idx.data_ptr(), B, pages.data_ptr(), k,
                                                 po.data_ptr(), PAGE, pl.data_ptr(), ps.data_ptr(), wsp.data_ptr(), wsp_n,
                                                 s) == 0

        t = one(reads, max(args.passes, 5))
        assert bool((ps == 0).all())
        pick = pages.long()
        assert torch.equal(po.view(k, PAGE), d.view(B, PAGE)[pick])
        res["page_reads"][f"{k}_requests"] = {"us_per_call": round(t * 1e6, 1), "gbs": gbs(k * PAGE, t)}
        del po, pl, ps, wsp
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
