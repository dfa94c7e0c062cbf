"""Guard-band canaries and reference error-code parity for the batched kernels.

GPU analogue of the reference's guard-page self tests (cl_tester.c:136-142, 196-218): every output
slot is pre-filled with a pattern, and after the launch the bytes the contract protects must be
untouched --
  decode    nothing at or past the block's capacity `cap` (inside the slot stride and in the next
            slot's guard band), on the staged path, the unstaged-input path and the global path,
            for valid, corrupted, truncated and under-sized streams;
  compress  nothing past csnappy_max_compressed_length(n) (the reference REQUIRES that much room and
            checks nothing, cl_tester.c:120-165 -- the kernel must not need more).
Also: corrupted streams that do NOT end inside a tag header are compared with the unmodified
reference's results (tests/golden/reference_cases.json), not only with the port -- only the
truncated-tag case is reference UB (SURVEY.md 0.5) and is defined here as -5.
"""
import hashlib

import numpy as np
import pytest

import oracle
from cases import CANARY_DECODE, corrupt_streams, fuzz_pages, reference_cases

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

PAT = 0xA5


@pytest.fixture(scope="module")
def cs():
    import csnappy_b200 as c

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    assert c.device_ok(), c.api.last_error()
    return c


@pytest.mark.parametrize("stage", [0, 2, 3, 4])
@pytest.mark.parametrize("lanes", [32, 16, 8])
@pytest.mark.parametrize("size,wm", [(4096, 13), (32768, 15)])
def test_decode_never_writes_at_or_past_cap(cs, lanes, stage, size, wm):
    streams, caps = corrupt_streams(oracle.best().compress_fragment, size, wm, *CANARY_DECODE[(size, wm)])
    ref = reference_cases()["canary_decode"][f"{size}/{wm}"]
    assert len(ref) == len(streams)
    B = len(streams)
    in_stride = (cs.csnappy_max_compressed_length(size) + 16 + 15) // 16 * 16
    out_stride = size + 256  # 256-byte guard band behind every slot
    host = np.zeros((B, in_stride), dtype=np.uint8)
    for i, s in enumerate(streams):
        host[i, : len(s)] = np.frombuffer(s, dtype=np.uint8)
    d_in = torch.from_numpy(host).cuda()
    d_len = torch.tensor([len(s) for s in streams], dtype=torch.int32).cuda()
    d_caps = torch.tensor(caps, dtype=torch.int32).cuda()
    out = torch.full((B * out_stride + 256,), PAT, dtype=torch.uint8, device="cuda")
    cs.set_tuning("decompress_lanes", lanes)
    cs.set_tuning("decompress_stage_input", stage)
    try:
        _, out_len, status = cs.batch_decompress(d_in, d_len, B, size, in_stride=in_stride, out_caps=d_caps,
                                                 out=out, out_stride=out_stride)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("decompress_lanes", 0)
        cs.set_tuning("decompress_stage_input", 0)
    o = out.cpu().numpy()
    ol, st = out_len.cpu().numpy(), status.cpu().numpy()
    assert (o[B * out_stride:] == PAT).all()
    n_err = 0
    for i, s in enumerate(streams):
        slot = o[i * out_stride:(i + 1) * out_stride]
        assert (slot[caps[i]:] == PAT).all(), (i, "wrote at or past cap", caps[i], int(st[i]))
        rc, exp = oracle.port().decompress_noheader(s, caps[i])
        assert st[i] == rc, (i, s.hex()[:60])
        if ref[i] is not None:  # None: the stream ends inside a tag header
            rrc, rsha = ref[i]
            assert (st[i], rc) == (rrc, rrc), (i, "differs from the unmodified reference", s.hex()[:60])
            if rrc == 0:
                assert hashlib.sha256(exp).hexdigest() == rsha
        if rc == 0:
            assert ol[i] == len(exp) and slot[: ol[i]].tobytes() == exp, i
        else:
            n_err += 1
    assert n_err >= B // 4


@pytest.mark.parametrize("lanes", [32, 16, 8])
@pytest.mark.parametrize("size,wm", [(4096, 13), (4096, 9), (32768, 15), (1000, 12)])
def test_compress_stays_inside_max_compressed_length(cs, lanes, size, wm):
    chk = oracle.best()
    pages = fuzz_pages(8800 + size + wm, 56 if size <= 4096 else 21, size)
    rng = np.random.default_rng(size)
    lens = [size if i % 3 else int(rng.integers(0, size + 1)) for i in range(len(pages))]
    B = len(pages)
    bound = [cs.csnappy_max_compressed_length(n) for n in lens]
    out_stride = (cs.csnappy_max_compressed_length(size) + 15) // 16 * 16 + 64
    host = np.zeros((B, size), dtype=np.uint8)
    for i, p in enumerate(pages):
        host[i, : lens[i]] = np.frombuffer(p[: lens[i]], dtype=np.uint8)
    d_in = torch.from_numpy(host).cuda()
    d_len = torch.tensor(lens, dtype=torch.int32).cuda()
    out = torch.full((B * out_stride + 256,), PAT, dtype=torch.uint8, device="cuda")
    cs.set_tuning("compress_lanes", lanes)
    try:
        _, out_len = cs.batch_compress_fragments(d_in, size, B, wm, in_len=d_len, out=out, out_stride=out_stride)
        torch.cuda.synchronize()
    finally:
        cs.set_tuning("compress_lanes", 0)
    o, ol = out.cpu().numpy(), out_len.cpu().numpy()
    assert (o[B * out_stride:] == PAT).all()
    for i in range(B):
        slot = o[i * out_stride:(i + 1) * out_stride]
        assert ol[i] <= bound[i]
        assert (slot[bound[i]:] == PAT).all(), (i, "wrote past csnappy_max_compressed_length", lens[i])
        assert slot[: ol[i]].tobytes() == chk.compress_fragment(host[i, : lens[i]].tobytes(), wm), i


def test_compress_refuses_oversized_lengths(cs):
    """d_in_len[i] above the stride / above 32768 is refused with the sentinel instead of being cut silently."""
    B, size = 8, 4096
    d_in = torch.zeros(B * size, dtype=torch.uint8, device="cuda")
    lens = torch.tensor([4096, 4097, 100, 40000, 0, 4096, 70000, 15], dtype=torch.int32).cuda()
    out, out_len = cs.batch_compress_fragments(d_in, size, B, 13, in_len=lens)
    torch.cuda.synchronize()
    ol = out_len.cpu().numpy().astype(np.uint32)
    assert [int(x) == 0xFFFFFFFF for x in ol] == [False, True, False, True, False, False, True, False]


def test_host_batch_decompress_rejects_length_beyond_stride(cs):
    B, stride = 4, 4816
    h_in = np.zeros((B, stride), dtype=np.uint8)
    h_len = np.array([10, stride + 1, 5, 5], dtype=np.uint32)
    back = np.zeros((B, 4096), dtype=np.uint8)
    blen = np.zeros(B, dtype=np.uint32)
    st = np.zeros(B, dtype=np.int32)
    rc = cs.api.lib().csnappy_batch_decompress_host(h_in.ctypes.data, stride, h_len.ctypes.data, B, back.ctypes.data,
                                                     4096, 4096, blen.ctypes.data, st.ctypes.data, 0)
    assert rc == cs.api.CSNAPPY_E_BAD_ARG
