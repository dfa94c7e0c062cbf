#!/usr/bin/env python
"""Regenerate tests/golden/ from the UNMODIFIED reference.

Needs the reference's sources (REF of oracle/Makefile) compiled by oracle/Makefile
into oracle/_ref/libcsnappy_ref.so:

    python tests/golden/make_golden.py           # everything below
    python tests/golden/make_golden.py --cases   # reference_cases.json alone

What it writes
  * gzip copies of the reference's own fixtures (data, not source):
    testdata/urls.10K, urls.10K.snappy, baddata3.snappy and the two
    unaligned_uint64_test files (reference Makefile:21-55 uses exactly these)
  * golden.json: outputs of the reference library on those fixtures and on
    seeded synthetic inputs -- sizes + sha256 of compressed streams for
    wm 9..16, per-fragment streams (4 KiB/13, 32 KiB/15, 32 KiB/16), the tiny
    input pins of SURVEY.md 8c, and the appendix-B decode matrix.
  * reference_cases.json: sha256 of the reference's results on the fuzz, edge-size and
    corrupted-stream inputs of tests/cases.py, as the tests compare them.  `--cases` records
    them with oracle.best() and names the checker in the file: without the reference library
    that is the port (oracle/snappy_oracle.c).
Tests read only what is committed here.
"""
import gzip
import hashlib
import json
import os
import shutil
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, ".."))
import oracle  # noqa: E402

REF_DATA = "/root/reference/testdata"


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def frag_stream(ref, data: bytes, block: int, wm: int):
    parts, total = [], 0
    for o in range(0, len(data), block):
        c = ref.compress_fragment(data[o:o + block], wm)
        parts.append(struct.pack("<I", len(c)) + c)
        total += len(c)
    return total, sha(b"".join(parts)), len(parts)


def synth_cases():
    """Seeded inputs reproducible from numpy alone (name -> bytes)."""
    rng = np.random.default_rng(0x5EED)
    cases = {}
    cases["random_4096"] = rng.integers(0, 256, 4096, dtype=np.uint8).tobytes()
    cases["zeros_4096"] = bytes(4096)
    for p in (1, 2, 3, 4, 5, 6, 7, 8, 13, 70):
        cases[f"period{p}_4096"] = bytes((i % p) for i in range(4096))
    cases["lowent_4096"] = rng.integers(0, 4, 4096, dtype=np.uint8).tobytes()
    cases["lowent_32768"] = rng.integers(0, 3, 32768, dtype=np.uint8).tobytes()
    words = [bytes(rng.integers(97, 123, int(rng.integers(2, 9)), dtype=np.uint8)) for _ in range(200)]
    text = b" ".join(words[int(i)] for i in rng.integers(0, 200, 9000))
    cases["words_32768"] = text[:32768]
    cases["words_4096"] = text[5000:5000 + 4096]
    for n in list(range(0, 21)) + [59, 60, 61, 62, 255, 256, 257, 258, 4081, 4095, 4097, 4111, 32753, 32767]:
        cases[f"words_len{n}"] = text[100:100 + n]
    return cases


def main():
    if not oracle.have_reference():
        oracle.build()
    ref = oracle.reference()
    os.makedirs(HERE, exist_ok=True)

    for name in ("urls.10K", "urls.10K.snappy", "baddata3.snappy"):
        with open(os.path.join(REF_DATA, name), "rb") as f, \
                gzip.GzipFile(os.path.join(HERE, name + ".gz"), "wb", mtime=0) as g:
            g.write(f.read())
    for name in ("unaligned_uint64_test.snappy.gz", "unaligned_uint64_test.bin.gz"):
        shutil.copyfile(os.path.join(REF_DATA, name), os.path.join(HERE, name))

    urls = open(os.path.join(REF_DATA, "urls.10K"), "rb").read()
    urls_snappy = open(os.path.join(REF_DATA, "urls.10K.snappy"), "rb").read()
    bad = open(os.path.join(REF_DATA, "baddata3.snappy"), "rb").read()
    uu_s = gzip.open(os.path.join(REF_DATA, "unaligned_uint64_test.snappy.gz")).read()
    uu_b = gzip.open(os.path.join(REF_DATA, "unaligned_uint64_test.bin.gz")).read()

    G = {"fixtures": {
        "urls.10K": {"len": len(urls), "sha256": sha(urls)},
        "urls.10K.snappy": {"len": len(urls_snappy), "sha256": sha(urls_snappy)},
        "baddata3.snappy": {"len": len(bad), "sha256": sha(bad)},
        "unaligned_uint64_test.snappy": {"len": len(uu_s), "sha256": sha(uu_s)},
        "unaligned_uint64_test.bin": {"len": len(uu_b), "sha256": sha(uu_b)},
    }}

    G["compress_urls"] = {}
    for wm in range(9, 17):
        c = ref.compress(urls, wm)
        G["compress_urls"][str(wm)] = {"len": len(c), "sha256": sha(c)}
    assert ref.compress(urls, 15) == urls_snappy, "fixture is not csnappy_compress(wm=15)"

    G["fragments_urls"] = {}
    for block, wm in ((4096, 13), (32768, 15), (32768, 16), (4096, 9), (4096, 16)):
        total, h, nb = frag_stream(ref, urls, block, wm)
        G["fragments_urls"][f"{block}/{wm}"] = {"blocks": nb, "total": total, "sha256": h}

    G["tiny"] = {}
    for label, data in [("a*%d" % n, b"a" * n) for n in (0, 1, 15, 16, 17, 20)] + [("abcd*10", b"abcd" * 10)]:
        G["tiny"][label] = {"input_hex": data.hex(), "wm16_hex": ref.compress(data, 16).hex()}

    G["synth"] = {}
    for name, data in synth_cases().items():
        ent = {"len": len(data), "in_sha256": sha(data)}
        for wm in (9, 13, 15, 16):
            c = ref.compress_fragment(data, wm)
            ent[f"frag_wm{wm}"] = {"len": len(c), "sha256": sha(c)}
        G["synth"][name] = ent

    # appendix-B decode matrix: (hex stream, capacity) -> reference result
    M = [
        ("", 100), ("08616263", 100), ("08616263", 2), ("10616263", 100),
        ("086162630100", 100), ("086162630104", 100), ("086162630103", 100),
        ("00611d01", 100), ("00611d01", 12), ("00611d01", 11),
        ("086162630f03000000", 100), ("086162630f03000080", 100),
        ("fcffffffff61", 100), ("fcffffff7f61", 100),
        ("c4666f6f6f6f6f6f", 50),
        ("0861626309" + "03", 100),
    ]
    G["decode_noheader"] = []
    for hx, cap in M:
        rc, out = ref.decompress_noheader(bytes.fromhex(hx), cap)
        G["decode_noheader"].append({"hex": hx, "cap": cap, "rc": rc, "out_hex": out.hex() if out is not None else None})

    H = [("0a08616263", 100), ("0208616263", 100), ("6408616263", 50), ("", 10), ("80", 10),
         ("808080808000", 10), ("32c4666f6f6f6f6f6f", 50)]
    G["decode_header"] = []
    for hx, dl in H:
        rc, _ = ref.decompress(bytes.fromhex(hx), dl)
        G["decode_header"].append({"hex": hx, "dst_len": dl, "rc": rc})

    V = ["", "80", "00", "7f", "8001", "ffffffff0f", "ffffffff7f", "8000", "808080808000", "87ed2a"]
    G["varint"] = []
    for hx in V:
        rc, val = ref.get_uncompressed_length(bytes.fromhex(hx))
        G["varint"].append({"hex": hx, "rc": rc, "value": val})

    rc, out = ref.decompress(bad, 130378)
    G["baddata3"] = {"rc": rc, "header_len": ref.get_uncompressed_length(bad)[1]}
    rc, out = ref.decompress(uu_s, len(uu_b))
    assert rc == 0 and out == uu_b
    G["unaligned_uint64"] = {"rc": rc, "out_sha256": sha(out)}

    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(G, f, indent=1, sort_keys=True)
    print("wrote", os.path.join(HERE, "golden.json"))
    write_reference_cases(ref)


def write_reference_cases(chk):
    """reference_cases.json: what tests/test_oracle.py and tests/test_gpu_canaries.py compare with."""
    from cases import (CANARY_DECODE, EDGE_COMPRESS_SIZES, EDGE_FRAGMENT_SIZES, corrupt_streams, corrupted_fragments,
                       edge_compress_input, edge_text, ends_inside_tag, ends_inside_tag_header, fuzz_pages)

    def result(rc, out):
        return [rc, None if out is None else sha(out)]

    R = {"checker": chk.kind}
    R["fuzz_fragments"] = {f"{size}/{wm}": [sha(chk.compress_fragment(p, wm)) for p in fuzz_pages(1234 + size + wm, 35, size)]
                           for size, wm in ((4096, 13), (4096, 9), (32768, 15), (32768, 16), (1000, 12), (20000, 14))}
    text = edge_text()
    R["edge_fragments"] = {str(wm): [sha(chk.compress_fragment(text[:n], wm)) for n in EDGE_FRAGMENT_SIZES]
                           for wm in (9, 13, 16)}
    R["edge_compress"] = {str(wm): [sha(chk.compress(edge_compress_input(text, n), wm)) for n in EDGE_COMPRESS_SIZES]
                          for wm in (9, 13, 15, 16)}
    # the reference's x86 path is undefined on a stream cut inside a tag's trailing bytes: recorded as None
    port = oracle.port()
    R["corruptions"] = [None if port.decompress_noheader(d, cap)[0] == oracle.E_DATA_MALFORMED and ends_inside_tag(d)
                        else result(*chk.decompress_noheader(d, cap)) for d, cap in corrupted_fragments(chk.compress_fragment)]
    pages = np.frombuffer(b"".join(fuzz_pages(77, 64, 4096)), dtype=np.uint8).reshape(64, 4096)
    out, out_len, _ = oracle.batch_compress(pages, 13, chk.kind, threads=2)
    R["bulk_4096_13"] = {"len": out_len.tolist(), "sha256": [sha(out[i, : out_len[i]].tobytes()) for i in range(64)]}
    R["canary_decode"] = {}
    for (size, wm), (seed, count) in CANARY_DECODE.items():
        streams, caps = corrupt_streams(chk.compress_fragment, size, wm, seed, count)
        R["canary_decode"][f"{size}/{wm}"] = [None if ends_inside_tag_header(s) else result(*chk.decompress_noheader(s, cap))
                                              for s, cap in zip(streams, caps)]
    path = os.path.join(HERE, "reference_cases.json")
    with open(path, "w") as f:
        json.dump(R, f, indent=0, sort_keys=True)
        f.write("\n")
    print("wrote", path, "checker", chk.kind)


if __name__ == "__main__":
    if "--cases" in sys.argv:
        write_reference_cases(oracle.best())
    else:
        main()
