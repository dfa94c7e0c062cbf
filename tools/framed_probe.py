"""Throughput of the framing-format calls on one GPU, device resident unless named otherwise, and of what a caller
without them has: csnappy_batch_compress + csnappy_batch_decompress(WITH_HEADER) over the same 64 KiB buffers (what
framing costs) and csnappy_compress + csnappy_stream_decompress of one buffer as a single stream.

    python tools/framed_probe.py [--gib 4] [--passes 3] [--out profiles/framed_probe.json]

Inputs are larger than L2 (4 GiB by default): text (32 MiB word-stream pool, 64 KiB windows at seeded offsets) and
mixed (zram-style 4 KiB pages: text / zero / random).  Every leg is warmed up once, then timed over --passes with CUDA
events; GB/s are of uncompressed bytes.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from csnappy_b200 import api, synth  # noqa: E402
from csnappy_b200._lib import lib  # noqa: E402

CHUNK = 65536


def timed(fn, passes):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(passes):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / passes


def gbs(n, t):
    return round(n / t / 1e9, 2)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable: {e}"
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name()}


def leg_class(d, passes):
    L = lib()
    s = torch.cuda.current_stream().cuda_stream
    n = d.numel()
    k = n // CHUNK
    res = {}
    cap = L.csnappy_framed_max_length(n)
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    olen = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = torch.empty(L.csnappy_framed_compress_workspace(n), dtype=torch.uint8, device="cuda")

    def comp():
        assert L.csnappy_framed_compress(d.data_ptr(), n, out.data_ptr(), cap, olen.data_ptr(), 16, ws.data_ptr(),
                                         ws.numel(), s) == 0

    res["framed_compress_gbs"] = gbs(n, timed(comp, passes))
    slen = int(olen.item())
    res["framed_ratio"] = round(slen / n, 4)
    del ws
    crc = torch.empty(k + 1, dtype=torch.int32, device="cuda")
    res["crc_kernel_gbs"] = gbs(n, timed(lambda: api.framed_crc32c_device(d, n, crc=crc), passes))
    dst = torch.empty(n, dtype=torch.uint8, device="cuda")
    r = torch.empty(4, dtype=torch.int64, device="cuda")
    wsd = torch.empty(L.csnappy_framed_decompress_workspace(slen), dtype=torch.uint8, device="cuda")
    walk = []

    def dec():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        assert L.csnappy_framed_decompress(out.data_ptr(), slen, dst.data_ptr(), n, r.data_ptr(), r.data_ptr() + 8,
                                           r.data_ptr() + 16, wsd.data_ptr(), wsd.numel(), s) == 0
        walk.append(time.perf_counter() - t0)  # the call returns after the walk, decoding enqueued

    res["framed_decompress_gbs"] = gbs(n, timed(dec, passes))
    assert int(r[0].item()) == n and int(r[1].item()) & 0xFFFFFFFF == 0 and torch.equal(dst, d)
    w = sorted(walk)[len(walk) // 2]
    res["walk_ms"] = round(w * 1e3, 3)
    res["walk_ns_per_chunk"] = round(w * 1e9 / max(k, 1), 1)
    res["walk_share_of_decompress"] = round(w / (n / (res["framed_decompress_gbs"] * 1e9)), 3)
    del wsd, dst, out
    torch.cuda.empty_cache()
    # the same 64 KiB buffers through the batched csnappy_compress / csnappy_decompress calls, without framing
    h_len = np.full(k, CHUNK, dtype=np.uint32)
    h_off = (np.arange(k, dtype=np.uint64) * np.uint64(CHUNK))
    stride = (5 + CHUNK + CHUNK // 6 + 64 + 15) // 16 * 16
    bout = torch.empty(k * stride, dtype=torch.uint8, device="cuda")
    blen = torch.empty(k, dtype=torch.int32, device="cuda")
    wsb_n = L.csnappy_batch_compress_workspace(h_len.ctypes.data, 0, k)
    wsb = torch.empty(wsb_n, dtype=torch.uint8, device="cuda")

    def bcomp():
        assert L.csnappy_batch_compress(d.data_ptr(), h_off.ctypes.data, 0, h_len.ctypes.data, 0, k, bout.data_ptr(),
                                        stride, blen.data_ptr(), 16, wsb.data_ptr(), wsb_n, s) == 0

    res["batch_compress_gbs"] = gbs(n, timed(bcomp, passes))
    del wsb
    bdst = torch.empty(n, dtype=torch.uint8, device="cuda")
    st = torch.empty(k, dtype=torch.int32, device="cuda")
    ol = torch.empty(k, dtype=torch.int32, device="cuda")

    def bdec():
        assert L.csnappy_batch_decompress(bout.data_ptr(), None, stride, blen.data_ptr(), k, bdst.data_ptr(), CHUNK,
                                          None, CHUNK, ol.data_ptr(), st.data_ptr(), api.BATCH_WITH_HEADER, s) == 0

    res["batch_decompress_with_header_gbs"] = gbs(n, timed(bdec, passes))
    assert torch.equal(bdst, d)
    del bout, bdst
    torch.cuda.empty_cache()
    return res


def leg_single_stream(d, passes):
    """csnappy_compress (host call) of one buffer, then its device-resident parallel stream decode."""
    n = d.numel()
    h = d.cpu().numpy()
    t0 = time.perf_counter()
    z = api.csnappy_compress(h.tobytes(), 16)
    tc = time.perf_counter() - t0
    rc, used = api.csnappy_get_uncompressed_length(z)
    src = torch.frombuffer(bytearray(z[rc:]), dtype=torch.uint8).cuda()
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    ws = torch.empty(lib().csnappy_stream_decompress_workspace(src.numel(), n), dtype=torch.uint8, device="cuda")
    res = torch.empty(2, dtype=torch.int32, device="cuda")
    t = timed(lambda: api.stream_decompress(src, src.numel(), n, out=out, workspace=ws, result=res), passes)
    assert torch.equal(out, d)
    return {"bytes": n, "csnappy_compress_host_gbs": gbs(n, tc), "stream_decompress_gbs": gbs(n, t)}


def leg_host(d, passes):
    """The host calls on pinned buffers (whole input staged, no H2D / kernel / D2H overlap)."""
    L = lib()
    n = d.numel()
    hin = d.cpu().pin_memory()
    cap = L.csnappy_framed_max_length(n)
    hout = torch.empty(cap, dtype=torch.uint8).pin_memory()
    hdst = torch.empty(n, dtype=torch.uint8).pin_memory()
    olen, dl = C.c_uint64(0), C.c_uint64(0)

    def run(fn):
        fn()
        t0 = time.perf_counter()
        for _ in range(passes):
            fn()
        return (time.perf_counter() - t0) / passes

    tc = run(lambda: L.csnappy_framed_compress_host(hin.data_ptr(), n, hout.data_ptr(), cap, C.byref(olen), 16))
    td = run(lambda: L.csnappy_framed_decompress_host(hout.data_ptr(), olen.value, hdst.data_ptr(), n, C.byref(dl), None))
    assert dl.value == n and torch.equal(hdst, hin)
    return {"bytes": n, "framed_compress_host_pinned_gbs": gbs(n, tc), "framed_decompress_host_pinned_gbs": gbs(n, td)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=4)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--out", default="profiles/framed_probe.json")
    a = ap.parse_args()
    n = int(a.gib * (1 << 30)) // CHUNK * CHUNK
    rep = {"card": card(), "bytes": n, "passes": a.passes, "classes": {}}
    for cls in ("text", "mixed"):
        d = synth.text_fragments(n // CHUNK, CHUNK) if cls == "text" else synth.mixed_pages(n // 4096, 4096)
        rep["classes"][cls] = leg_class(d, a.passes)
        print(cls, json.dumps(rep["classes"][cls]), flush=True)
        if cls == "text":
            small = d[: min(n, 1 << 30)].clone()
            del d
            torch.cuda.empty_cache()
            rep["single_stream_text"] = leg_single_stream(small, a.passes)
            print("single", json.dumps(rep["single_stream_text"]), flush=True)
            rep["host_text"] = leg_host(small, a.passes)
            print("host", json.dumps(rep["host_text"]), flush=True)
            del small
        else:
            del d
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rep, f, indent=1)
    print(json.dumps(rep))


if __name__ == "__main__":
    main()
