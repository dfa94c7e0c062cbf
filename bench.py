#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native csnappy hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--pages P]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], "zram-style batch", as defined in SURVEY.md 8d config 2): per GPU
1 Mi synthetic 4 KiB pages, class per page from splitmix64(seed ^ index): 50 % text (a 4096-byte slice
of the reference's urls.10K corpus at a seeded offset; --text words switches to the purely synthetic
Zipf word stream, which is also reported as `alt_workload`), 25 % zero, 25 % random
(csnappy_b200/synth.py), csnappy_compress_fragment
semantics with workmem_bytes_power_of_two = 13, then csnappy_decompress_noheader of the result.
One STEP = compress the whole batch + decompress the whole batch.  Metric: GB/s of UNCOMPRESSED
bytes through the codec = (bytes compressed + bytes decompressed) / step time, whole job
(sum over ranks, max time over ranks).  Pages are independent, so ranks shard the page range
with no data-path collective ("weak": per-GPU batch fixed); NCCL is used for the barrier and
the max-over-ranks only.

`value`      device-resident: inputs already in HBM, CUDA events around K steps.
`e2e`        same metric through the host-buffer C-ABI (csnappy_bc_compress_host + csnappy_bc_decompress_host, the
             block_compressor page container) with pinned host buffers: H2D of every page and D2H of every
             result inside the timed region.
`e2e_concurrent` (N = 1) the two calls running in two threads at once (both PCIe directions busy).
`e2e_pageable`   (N = 1) the same calls on ordinary (pageable) caller memory.
`roofline`   dominant kernel (compress) against the measured HBM copy peak;
             algorithmic bytes = sum N_in + sum C_out + 4 B (SURVEY.md 8d).
`workloads`  BASELINE.json configs[2] and [3], device-resident, every rank, reduced like `value`:
             fragments_32k (32 KiB text fragments, wm 15 and 16, 4 GiB per GPU, seed 0x5EED0002) and decode_only
             (a pre-compressed corpus of 64 GiB per GPU in 16 GiB waves, 4 KiB mixed pages and 32 KiB text
             fragments, seed 0x5EED0003), each with its own roofline fraction and a sample checked against the CPU reference.
`cpu_baseline` the unmodified reference (oracle/_ref) or the oracle port on this box's cores.
--impl reference times that CPU implementation alone (same config, same protocol: oracle.BatchRunner.measure).
--dump-outputs DIR writes what the last timed step returned (rank 0's pages) as .npy files, see dump_outputs();
             the inputs depend on the arguments only, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PAGE = 4096
WM = 13
SEED = 0x5EED0001
METRIC = "compress+decompress throughput, GB/s of uncompressed data, 4 KiB pages (wm 13)"
TEXT_DESC = {"urls": "4096-byte slices of the reference's urls.10K at seeded offsets",
             "words": "Zipf(1.1) word stream over a 4096-word vocabulary"}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.idx), "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx = float(c[2])
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


def workload_config(text: str, pages: int, world: int, ratio):
    """`config` of the JSON line -- the SAME dict in both arms (the driver compares them)."""
    return {"workload": f"zram-style batch: synthetic 4 KiB pages (50% text [{TEXT_DESC[text]}] / 25% zero / "
                        "25% random), wm 13, compress then decompress", "pages_per_gpu": pages, "page_bytes": PAGE,
            "wm": WM, "ratio": ratio, "parallelism": f"shard{world} (no collective)",
            "l2": "inputs (4 GiB per GPU) exceed the 126 MB L2; no explicit flush",
            "value_definition": "(bytes compressed + bytes decompressed) / step time"}


def cpu_measure(host_units, wm: int, warmup: int, steps: int):
    """The one CPU-baseline protocol (both arms): the reference's codec on all host cores over `host_units`
    [S, unit], buffers allocated and touched once, mean of `steps` passes after `warmup` passes.
    -> (runner, compress_s, decompress_s, impl, cores)"""
    import oracle

    impl = "reference" if oracle.have_reference() else "port"
    cores = host_cores()
    r = oracle.BatchRunner(host_units, wm, impl, threads=cores)
    tc, td = r.measure(warmup, steps)
    return r, tc, td, impl, cores


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's own CPU implementation on this box's cores, on rank 0's shard of the
    same workload (all `--pages` pages per step unless --cpu-pages bounds the sample)."""
    if rank != 0:
        return
    import torch

    from csnappy_b200 import synth

    S = min(args.pages, args.cpu_pages) if args.cpu_pages else args.pages
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    pages = synth.mixed_pages(S, PAGE, seed=SEED, device=dev, text=args.text).view(S, PAGE).cpu().numpy()
    r, tc, td, impl, cores = cpu_measure(pages, WM, args.warmup, args.steps)
    value = 2 * S * PAGE / (tc + td) / 1e9
    ratio = round(float(r.comp_len.sum(dtype="uint64")) / (S * PAGE), 4)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * (tc + td), 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.text, args.pages, args.gpus, ratio),
        "compress_gbs": round(S * PAGE / tc / 1e9, 3), "decompress_gbs": round(S * PAGE / td / 1e9, 3),
        "cpu_baseline": {"value": round(value, 3), "unit": "GB/s", "cores": cores, "kind": impl,
                         "sample": f"{S} pages ({S * PAGE >> 20} MiB) per step = rank 0's shard, compress + decompress, "
                                   f"{cores} pthreads, static partition, mean of {args.steps} steps after {args.warmup} warm-ups"},
        "e2e": {"value": round(value, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def dump_outputs(path: str, B: int, ostride: int, comp, comp_len, back, back_len, status):
    """The results of the timed step as float32 .npy files under `path` (57 MB at most), on pages picked by a fixed
    seed: compressed_len / decompressed_len / status of up to 1 Mi pages (all pages of the default batch; their
    indices in len_pages.npy) and compressed / decompressed bytes of 1024 pages (indices in byte_pages.npy).  A
    compressed slot is zeroed past its length: those bytes are not part of the result."""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0x5EED0D)
    len_pages = np.sort(rng.choice(B, min(B, 1 << 20), replace=False))
    byte_pages = np.sort(rng.choice(B, min(B, 1024), replace=False))
    li = torch.from_numpy(len_pages).to(comp.device)
    bi = torch.from_numpy(byte_pages).to(comp.device)
    c = comp.view(B, ostride).index_select(0, bi).float()
    c *= torch.arange(ostride, device=c.device)[None, :] < comp_len.index_select(0, bi)[:, None]
    out = {"len_pages": len_pages.astype(np.float64), "byte_pages": byte_pages.astype(np.float64),
           "compressed_len": comp_len.index_select(0, li), "decompressed_len": back_len.index_select(0, li),
           "status": status.index_select(0, li), "compressed": c,
           "decompressed": back.view(B, PAGE).index_select(0, bi)}
    for name, a in out.items():
        if isinstance(a, torch.Tensor):
            a = a.float().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a)


def run_workloads(args, cs, synth, dev, rank, world, barrier):
    """BASELINE.json configs[2] "32 KB fragments over a text-like stream" and configs[3] "decompression-only throughput
    of a pre-compressed corpus" (SURVEY.md 8d configs 3 and 4).  Weak scaling like the main workload: every rank owns
    its own range of the global fragment / page sequence.  Times are CUDA events on the launching stream, max over
    ranks; bytes are summed over ranks.  Each shape is checked: exact round trip of everything, and the compressed
    bytes of a sample against the CPU reference (oracle/, the checker -- never the thing timed)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import oracle

    peak, _ = measured_peak()
    impl = "reference" if oracle.have_reference() else "port"
    FRAG = 32768

    def timed(fn, reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def reduce(ms_list, sums):
        v = torch.tensor(ms_list, dtype=torch.float64, device=dev)
        t = torch.tensor(sums, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return v.tolist(), t.tolist()

    def check_sample(units2d, unit, wm, comp, comp_len, ostride, k=64):
        """compressed bytes of k units spread over the batch == the CPU reference's"""
        n = units2d.shape[0]
        idx = np.unique(np.linspace(0, n - 1, k).astype(np.int64))
        ti = torch.from_numpy(idx).to(dev)
        host = units2d.index_select(0, ti).cpu().numpy()
        r = oracle.BatchRunner(host, wm, impl, threads=min(host_cores(), len(idx)))
        r.compress()
        got_len = comp_len.index_select(0, ti).cpu().numpy().astype(np.uint32)
        got = comp.view(n, ostride).index_select(0, ti).cpu().numpy()
        assert (got_len == r.comp_len).all(), "compressed sizes differ from the CPU reference"
        for j in range(len(idx)):
            assert got[j, : got_len[j]].tobytes() == r.compressed(j), f"compressed bytes of unit {idx[j]} differ"
        return len(idx)

    def codec_pass(data, unit, n, wm, reps_c, reps_d, bufs):
        """compress (timed reps_c times) + decompress (timed reps_d times) of n units; -> ms_c, ms_d, csum"""
        comp, comp_len, back, back_len, status, ostride = bufs
        cfn = lambda: cs.batch_compress_fragments(data, unit, n, wm, out=comp, out_len=comp_len, out_stride=ostride)
        dfn = lambda: cs.batch_decompress(comp, comp_len, n, unit, in_stride=ostride, out=back, out_stride=unit,
                                          out_len=back_len, status=status)
        cfn()  # warm-up; also what the decoder reads
        ms_c = timed(cfn, reps_c) if reps_c else None
        dfn()
        ms_d = timed(dfn, reps_d)
        assert int((status[:n] != 0).sum()) == 0 and int((back_len[:n] != unit).sum()) == 0
        assert torch.equal(back[: n * unit], data), "round trip mismatch"
        return ms_c, ms_d, float(comp_len[:n].sum(dtype=torch.int64))

    def alloc(unit, n):
        ostride = cs.api.out_stride_for(unit)
        return (torch.empty(n * ostride, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                torch.empty(n * unit, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.int32, device=dev),
                torch.empty(n, dtype=torch.int32, device=dev), ostride)

    out = {}
    # ---- fragments_32k: block_compressor / csnappy_compress fragments of a text-like stream -------------------------
    n = max(1, int(args.frag_gib * (1 << 30)) // FRAG)
    data = synth.text_fragments(n, FRAG, seed=0x5EED0002, device=dev, first=rank * n)
    bufs = alloc(FRAG, n)
    frag = {"unit_bytes": FRAG, "units_per_gpu": n, "seed": "0x5EED0002",
            "data": "32 KiB slices of the Zipf word stream at seeded offsets (synth.text_fragments)"}
    for wm in (15, 16):
        ms_c, ms_d, csum = codec_pass(data, FRAG, n, wm, 2, 3, bufs)
        checked = check_sample(data.view(n, FRAG), FRAG, wm, bufs[0], bufs[1], bufs[5])
        (ms_c, ms_d), (tot_n, tot_c) = reduce([ms_c, ms_d], [float(n) * FRAG, csum])
        alg_c, alg_d = n * FRAG + tot_c / world + 4 * n, tot_c / world + n * FRAG + 8 * n
        frag[f"wm{wm}"] = {"ratio": round(tot_c / tot_n, 4),
                           "compress_gbs": round(tot_n / ms_c / 1e6, 2), "decompress_gbs": round(tot_n / ms_d / 1e6, 2),
                           "compress_ms": round(ms_c, 3), "decompress_ms": round(ms_d, 3),
                           "roofline_frac_compress": round(alg_c / ms_c / 1e6 / peak, 4),
                           "roofline_frac_decompress": round(alg_d / ms_d / 1e6 / peak, 4),
                           "units_checked_against_cpu_reference": checked}
    out["fragments_32k"] = frag
    del data, bufs
    torch.cuda.empty_cache()

    # ---- decode_only: a pre-compressed corpus, decoded in waves ---------------------------------------------------
    # The corpus is compressed on the device by the kernels whose output is byte-identical to the reference's
    # (tests/, and the per-wave sample check below); only the decode passes are timed.
    dec = {"seed": "0x5EED0003", "corpus_gib_per_gpu": args.decode_gib, "wave_gib": args.wave_gib}
    for name, unit, wm in (("pages_4k", PAGE, WM), ("fragments_32k", FRAG, 15)):
        wave_units = max(1, int(args.wave_gib * (1 << 30)) // unit)
        waves = max(1, int(round(args.decode_gib / args.wave_gib)))
        bufs = alloc(unit, wave_units)
        ms_sum, n_sum, c_sum, checked = 0.0, 0.0, 0.0, 0
        for w in range(waves):
            first = (rank * waves + w) * wave_units
            if unit == PAGE:
                data = synth.mixed_pages(wave_units, PAGE, seed=0x5EED0003, device=dev, first_page=first, text=args.text)
            else:
                data = synth.text_fragments(wave_units, FRAG, seed=0x5EED0003, device=dev, first=first)
            _, ms_d, csum = codec_pass(data, unit, wave_units, wm, 0, 3, bufs)
            checked += check_sample(data.view(wave_units, unit), unit, wm, bufs[0], bufs[1], bufs[5], k=32)
            ms_sum, n_sum, c_sum = ms_sum + ms_d, n_sum + float(wave_units) * unit, c_sum + csum
            del data
        (ms_d,), (tot_n, tot_c) = reduce([ms_sum], [n_sum, c_sum])
        alg_d = (tot_c + tot_n) / world + 8 * wave_units * waves
        dec[name] = {"unit_bytes": unit, "wm": wm, "units_per_wave": wave_units, "waves": waves,
                     "bytes_decoded_per_gpu": int(n_sum), "ratio": round(tot_c / tot_n, 4),
                     "decompress_gbs": round(tot_n / ms_d / 1e6, 2), "decompress_ms_per_corpus": round(ms_d, 3),
                     "roofline_frac_decompress": round(alg_d / ms_d / 1e6 / peak, 4),
                     "units_checked_against_cpu_reference": checked,
                     "note": "slot and output offsets of a wave exceed 2^32; every wave is checked by exact round trip"}
        del bufs
        torch.cuda.empty_cache()
    out["decode_only"] = dec
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pages", type=int, default=1 << 20, help="pages per GPU (default 1 Mi = 4 GiB)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--lanes-c", type=int, default=0)
    ap.add_argument("--lanes-d", type=int, default=0)
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--stage-d", type=int, default=0)
    ap.add_argument("--smem-d", type=int, default=0)
    ap.add_argument("--text", default="urls", choices=["urls", "words"],
                    help="text class (SURVEY.md 8d config 2): 4 KiB slices of the reference's urls.10K at seeded "
                         "offsets (default), or the purely synthetic alternative, a Zipf(1.1) word stream")
    ap.add_argument("--no-alt", action="store_true", help="skip the short run on the alternative text class")
    ap.add_argument("--cpu-pages", type=int, default=0, help="--impl reference: bound the pages per step (0 = all --pages)")
    ap.add_argument("--no-workloads", action="store_true", help="skip the fragments_32k / decode_only workloads")
    ap.add_argument("--frag-gib", type=float, default=4.0, help="fragments_32k: GiB of 32 KiB fragments per GPU")
    ap.add_argument("--decode-gib", type=float, default=64.0, help="decode_only: GiB of corpus per GPU and unit size")
    ap.add_argument("--wave-gib", type=float, default=16.0, help="decode_only: GiB per wave")
    ap.add_argument("--only", default="", choices=["", "text", "zero", "random"],
                    help="diagnostic: make every page of one class (not the BASELINE workload)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed (rank 0's pages) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import csnappy_b200 as cs
    from csnappy_b200 import shard, synth

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert cs.device_ok(), cs.api.last_error()
    if args.lanes_c:
        cs.set_tuning("compress_lanes", args.lanes_c)
    if args.lanes_d:
        cs.set_tuning("decompress_lanes", args.lanes_d)
    if args.ctas_per_sm:
        cs.set_tuning("ctas_per_sm", args.ctas_per_sm)
    if args.stage_d:
        cs.set_tuning("decompress_stage_input", args.stage_d)
    if args.smem_d:
        cs.set_tuning("decompress_smem_kb", args.smem_d)

    B = args.pages
    first, _ = shard.block_range(B * world, rank, world)  # weak scaling: rank r owns pages [r*B, (r+1)*B)
    pages = synth.mixed_pages(B, PAGE, seed=SEED, device=dev, first_page=first, only=args.only, text=args.text)
    ostride = cs.api.out_stride_for(PAGE)
    comp = torch.empty(B * ostride, dtype=torch.uint8, device=dev)
    comp_len = torch.empty(B, dtype=torch.int32, device=dev)
    back = torch.empty(B * PAGE, dtype=torch.uint8, device=dev)
    back_len = torch.empty(B, dtype=torch.int32, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)

    def step(ev=None):
        if ev:
            ev[0].record()
        cs.batch_compress_fragments(pages, PAGE, B, WM, out=comp, out_len=comp_len, out_stride=ostride)
        if ev:
            ev[1].record()
        cs.batch_decompress(comp, comp_len, B, PAGE, in_stride=ostride, out=back, out_stride=PAGE,
                            out_len=back_len, status=status)
        if ev:
            ev[2].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    # correctness of what is being timed: exact round trip + all-OK status
    assert int((status != 0).sum()) == 0 and int((back_len != PAGE).sum()) == 0
    assert torch.equal(back, pages), "round trip mismatch"
    csum = int(comp_len.sum())

    sampler = ClockSampler(local_rank)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = cs.kernel_launches()
    barrier()
    if rank == 0:
        sampler.start()
    t0.record()
    for k in range(args.steps):
        step(evs[k])
    t1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = cs.kernel_launches() - launches0
    elapsed_ms = t0.elapsed_time(t1)
    tc_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)
    td_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in evs)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, B, ostride, comp, comp_len, back, back_len, status)

    # ---- e2e through the host-buffer C-ABI with pinned host memory ------------------------
    # The call a block_compressor / zram style user makes: pages in host memory -> the page container
    # (block_compressor.c:275-345) in host memory, and back (block_compressor.c:347-394).  Every step
    # copies all pages H2D, the container D2H, the container H2D and all pages D2H inside the timed region.
    e2e_ms = e2e_pageable_ms = e2e_both_ms = None
    h2d = d2h = 0
    if not args.no_e2e:
        h_in = torch.empty(B * PAGE, dtype=torch.uint8, pin_memory=True)
        h_cont = torch.empty(cs.api.bc_max_container_length(B * PAGE, PAGE), dtype=torch.uint8, pin_memory=True)
        h_back = torch.empty(B * PAGE, dtype=torch.uint8, pin_memory=True)
        h_in.copy_(pages)
        torch.cuda.synchronize()
        clen_box = [0]

        def e2e_step():
            ta = time.perf_counter()
            clen_box[0] = cs.api.bc_compress_host(h_in, B * PAGE, h_cont, WM, PAGE)
            tb = time.perf_counter()
            rc, olen, _ = cs.api.bc_decompress_host(h_cont, clen_box[0], h_back, PAGE)
            if os.environ.get("CSB_BENCH_DEBUG"):
                print(f"e2e compress {1e3 * (tb - ta):.1f} ms decompress {1e3 * (time.perf_counter() - tb):.1f} ms",
                      file=sys.stderr, flush=True)
            assert rc == 0 and olen == B * PAGE

        e2e_step()
        assert torch.equal(h_back, h_in), "e2e round trip mismatch"
        e2e_step()  # second warm-up: staging buffers have their final size now
        n_e2e = max(3, min(args.steps, 10))
        barrier()
        w0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        torch.cuda.synchronize()
        e2e_ms = 1e3 * (time.perf_counter() - w0) / n_e2e
        payload = clen_box[0] - 4 - 4 * B
        h2d = B * PAGE + payload + 4 * B
        d2h = payload + 4 * B + 8 * ((B + 8191) // 8192) + B * PAGE + 8 * B
        if world == 1:  # single-GPU runs only: the extra host buffers and copy threads of 8 ranks would fight over one host
            # both directions of the bus at once: one thread compresses the batch while another decompresses the
            # container of the previous step (the calls are re-entrant; a zram-like user runs both all the time).
            # Same work per step as `e2e`, but H2D and D2H are balanced instead of 4.3 GB one way + 2.4 GB the other.
            import threading

            h_cont2 = torch.empty(h_cont.numel(), dtype=torch.uint8, pin_memory=True)

            def both_step():
                def comp():
                    assert cs.api.bc_compress_host(h_in, B * PAGE, h_cont2, WM, PAGE) == clen_box[0]

                t = threading.Thread(target=comp)
                t.start()
                rc, olen, _ = cs.api.bc_decompress_host(h_cont, clen_box[0], h_back, PAGE)
                t.join()
                assert rc == 0 and olen == B * PAGE

            both_step()
            barrier()
            w0 = time.perf_counter()
            for _ in range(3):
                both_step()
            torch.cuda.synchronize()
            e2e_both_ms = 1e3 * (time.perf_counter() - w0) / 3
            assert torch.equal(h_cont2[: clen_box[0]], h_cont[: clen_box[0]]) and torch.equal(h_back, h_in)
            del h_cont2
            # the same calls on ordinary pageable caller memory (what a caller that never heard of CUDA passes in)
            p_in, p_back = h_in.clone(memory_format=torch.contiguous_format), torch.empty(B * PAGE, dtype=torch.uint8)
            p_cont = torch.empty(h_cont.numel(), dtype=torch.uint8)
            assert not p_in.is_pinned() and not p_cont.is_pinned()
            h_in, h_cont, h_back = p_in, p_cont, p_back
            e2e_step()
            assert torch.equal(h_back, h_in), "pageable e2e round trip mismatch"
            barrier()
            w0 = time.perf_counter()
            for _ in range(2):
                e2e_step()
            torch.cuda.synchronize()
            e2e_pageable_ms = 1e3 * (time.perf_counter() - w0) / 2
            del p_in, p_cont, p_back
        del h_in, h_cont, h_back

    # ---- short diagnostic runs (device-resident, rank 0's times): the alternative text class of SURVEY 8d, and
    # ---- every page class of the main workload on its own (SURVEY 8d: "report per-class and mixed") ----------
    alt = per_class = None
    if not args.no_alt and not args.only:
        Ba = min(B, 1 << 18)
        a_comp = torch.empty(Ba * ostride, dtype=torch.uint8, device=dev)
        a_len = torch.empty(Ba, dtype=torch.int32, device=dev)
        a_back = torch.empty(Ba * PAGE, dtype=torch.uint8, device=dev)
        a_blen = torch.empty(Ba, dtype=torch.int32, device=dev)
        a_st = torch.empty(Ba, dtype=torch.int32, device=dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

        def short_run(pa, n):
            def one(record):
                if record:
                    ev[0].record()
                cs.batch_compress_fragments(pa, PAGE, n, WM, out=a_comp, out_len=a_len, out_stride=ostride)
                if record:
                    ev[1].record()
                cs.batch_decompress(a_comp, a_len, n, PAGE, in_stride=ostride, out=a_back, out_stride=PAGE,
                                    out_len=a_blen, status=a_st)
                if record:
                    ev[2].record()

            for _ in range(3):
                one(False)
            tc, td = [], []
            for _ in range(3):
                one(True)
                torch.cuda.synchronize()
                tc.append(ev[0].elapsed_time(ev[1]))
                td.append(ev[1].elapsed_time(ev[2]))
            assert int((a_st[:n] != 0).sum()) == 0 and torch.equal(a_back[: n * PAGE], pa)
            tc, td = statistics.mean(tc) * 1e-3, statistics.mean(td) * 1e-3
            return {"pages_per_gpu": n, "ratio": round(float(a_len[:n].sum()) / (n * PAGE), 4),
                    "compress_gbs": round(world * n * PAGE / tc / 1e9, 2),
                    "decompress_gbs": round(world * n * PAGE / td / 1e9, 2),
                    "value": round(2 * world * n * PAGE / (tc + td) / 1e9, 2)}

        other = "words" if args.text == "urls" else "urls"
        alt = {"text": TEXT_DESC[other], "note": "rank 0's times, mean of 3 steps after 3 warm-ups",
               **short_run(synth.mixed_pages(Ba, PAGE, seed=SEED, device=dev, first_page=first, text=other), Ba)}
        Bc = min(B, 1 << 18)  # enough pages for the default decoder routing of a large batch (lane per page)
        per_class = {c: short_run(synth.mixed_pages(Bc, PAGE, seed=SEED, device=dev, first_page=first, text=args.text,
                                                     only=c), Bc) for c in ("text", "zero", "random")}
        del a_comp, a_back

    # ---- BASELINE.json configs[2] and [3] (SURVEY.md 8d configs 3 and 4), device-resident, every rank ---------
    workloads = None
    S_cpu = min(B, 1 << 18)
    host_sample = got_len_sample = None
    if world == 1 and not args.no_cpu:
        host_sample = pages.view(B, PAGE)[:S_cpu].cpu().numpy()
        got_len_sample = comp_len[:S_cpu].cpu().numpy().astype(np.uint32)
    if not args.no_workloads and not args.only:
        del pages, comp, back
        torch.cuda.empty_cache()
        workloads = run_workloads(args, cs, synth, dev, rank, world, barrier)

    # ---- reduce over ranks: max time, sum bytes -------------------------------------------
    vals = torch.tensor([elapsed_ms, tc_ms, td_ms, e2e_ms or 0.0, e2e_pageable_ms or 0.0, e2e_both_ms or 0.0], dtype=torch.float64, device=dev)
    sums = torch.tensor([float(B * PAGE), float(csum), float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    elapsed_ms, tc_ms, td_ms, e2e_max, e2e_pageable_max, e2e_both_max = vals.tolist()
    total_n, total_c, total_launches = sums.tolist()

    if rank == 0:
        ms_per_step = elapsed_ms / args.steps
        value = 2 * total_n / (ms_per_step * 1e-3) / 1e9
        peak, peak_src = measured_peak()
        # roofline of the dominant kernel, per launch on ONE GPU (rank 0's kernel times are the max over ranks)
        alg_c = B * PAGE + total_c / world + 4 * B
        alg_d = total_c / world + B * PAGE + 8 * B
        ach_c = alg_c / (tc_ms * 1e-3) / 1e9
        ach_d = alg_d / (td_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f)
        dominant = "compress" if tc_ms >= td_ms else "decompress"
        # large batches decode with one lane per page (decompress_lane_kernel), smaller ones with a warp per page
        kname = {"compress": "compress_kernel", "decompress": "decompress_lane_kernel" if B >= 148 * 1100 else "decompress_kernel"}
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.text, B, world, round(total_c / total_n, 4)),
            "compress_gbs": round(total_n / (tc_ms * 1e-3) / 1e9, 2),
            "decompress_gbs": round(total_n / (td_ms * 1e-3) / 1e9, 2),
            "roofline": {"kernel": kname[dominant], "bound": "hbm",
                         "achieved": round(ach_c if dominant == "compress" else ach_d, 2), "peak": peak,
                         "unit": "GB/s", "frac": round((ach_c if dominant == "compress" else ach_d) / peak, 4),
                         "traffic": (int((traffic or {}).get(dominant) * B / traffic["pages"]) if traffic else None),
                         "traffic_source": ("profiles/traffic.json: ncu dram bytes of one launch at "
                                            f"{traffic['pages']} pages, scaled to this batch") if traffic else None,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(alg_c if dominant == "compress" else alg_d),
                         "kernel_ms": round(tc_ms if dominant == "compress" else td_ms, 3)},
            "roofline_other": {"kernel": kname["decompress" if dominant == "compress" else "compress"],
                               "achieved": round(ach_d if dominant == "compress" else ach_c, 2),
                               "frac": round((ach_d if dominant == "compress" else ach_c) / peak, 4),
                               "kernel_ms": round(td_ms if dominant == "compress" else tc_ms, 3)},
            "gpu_launches": int(total_launches),
            "clocks": clocks,
        }
        if alt:
            line["alt_workload"] = alt
            line["per_class"] = per_class
        if e2e_max:
            line["e2e"] = {"value": round(2 * total_n / (e2e_max * 1e-3) / 1e9, 2), "unit": "GB/s",
                           "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world,
                           "ms_per_step": round(e2e_max, 2),
                           "api": "csnappy_bc_compress_host + csnappy_bc_decompress_host (block_compressor page container), pinned host buffers"}
        if e2e_both_max:
            line["e2e_concurrent"] = {"value": round(2 * total_n / (e2e_both_max * 1e-3) / 1e9, 2), "unit": "GB/s",
                                      "ms_per_step": round(e2e_both_max, 2),
                                      "api": "csnappy_bc_compress_host of the batch and csnappy_bc_decompress_host of the previous "
                                             "container running in two threads at once (pinned buffers): both PCIe directions busy"}
        if e2e_pageable_max:
            line["e2e_pageable"] = {"value": round(2 * total_n / (e2e_pageable_max * 1e-3) / 1e9, 2), "unit": "GB/s",
                                    "ms_per_step": round(e2e_pageable_max, 2),
                                    "api": "the same two calls on pageable caller memory (chunks staged through pinned slot buffers by the "
                                           "library's copy threads), mean of 2 steps after 1 warm-up"}
        if workloads:
            line["workloads"] = workloads
        if host_sample is not None:
            r, tc, td, impl, cores = cpu_measure(host_sample, WM, 1, 3)
            r1 = __import__("oracle").BatchRunner(host_sample[: S_cpu // 8], WM, impl, threads=1)
            t1c = r1.compress()
            # the same pass is the bulk parity check of what was timed
            assert (got_len_sample == r.comp_len).all(), "GPU compressed sizes differ from the CPU reference"
            line["cpu_baseline"] = {
                "value": round(2 * S_cpu * PAGE / (tc + td) / 1e9, 3), "unit": "GB/s", "cores": cores, "kind": impl,
                "sample": f"first {S_cpu} pages ({S_cpu * PAGE >> 20} MiB) of the same batch, compress + decompress, "
                          f"{cores} pthreads, static partition, mean of 3 steps after 1 warm-up",
                "compress_gbs": round(S_cpu * PAGE / tc / 1e9, 3), "decompress_gbs": round(S_cpu * PAGE / td / 1e9, 3),
                "single_thread_compress_gbs": round((S_cpu // 8) * PAGE / t1c / 1e9, 3)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
