"""The batched framing calls at the C-ABI boundary without a GPU: the workspace arithmetic, and the calls failing
loudly (CSNAPPY_E_DEVICE) rather than falling back when no device is present."""
import ctypes as C

import numpy as np
import pytest

SLOT = 38272  # fragment slot of the writer: csnappy_max_compressed_length(32768) rounded up to 16
NONE = 2**64 - 1


@pytest.fixture(scope="module")
def lib():
    from csnappy_b200 import build

    build.build()
    from csnappy_b200._lib import lib as load

    return load()


def u64(xs):
    return np.ascontiguousarray(np.asarray(xs, dtype=np.uint64))


def compress_ws(lib, lens):
    a = u64(lens)
    return lib.csnappy_framed_batch_compress_workspace(a.ctypes.data if a.size else None, len(a))


def decompress_ws(lib, lens):
    a = u64(lens)
    return lib.csnappy_framed_batch_decompress_workspace(a.ctypes.data if a.size else None, len(a))


def single_tables(n):
    """Table parts of one single call's workspace, without alignment: writer fragment slots + fragment sizes, CRCs,
    record sizes and offsets; reader result words + the per-chunk tables."""
    frags, chunks = -(-n // 32768), -(-n // 65536)
    return frags * SLOT + frags * 4 + chunks * 8 + (chunks + 1) * 8, 32 + 56 * (n // 8 + 1)


def test_workspace_covers_the_single_calls_and_is_monotone(lib):
    rng = np.random.default_rng(1)
    for trial in range(40):
        lens = [int(x) for x in rng.choice([0, 1, 7, 8, 4096, 32767, 32768, 32769, 65536, 65537, int(rng.integers(0, 10**7))],
                                           int(rng.integers(1, 30)))]
        wc, wd = compress_ws(lib, lens), decompress_ws(lib, lens)
        assert wc >= sum(single_tables(n)[0] for n in lens), lens
        assert wd >= sum(single_tables(n)[1] for n in lens), lens
        i = int(rng.integers(0, len(lens)))
        for more in (1, 8, 32768, 65536):
            grown = lens[:i] + [lens[i] + more] + lens[i + 1:]
            assert compress_ws(lib, grown) >= wc and decompress_ws(lib, grown) >= wd, (lens, i, more)
        assert compress_ws(lib, lens + [0]) >= wc and decompress_ws(lib, lens + [0]) >= wd
    assert compress_ws(lib, []) > 0 and decompress_ws(lib, []) > 0


def test_workspace_beyond_the_limits(lib):
    assert compress_ws(lib, [(2**32 - 2) * 32768]) < NONE
    assert compress_ws(lib, [(2**32 - 2) * 32768 + 1]) == NONE
    assert compress_ws(lib, [2**31 * 32768, 2**31 * 32768]) == NONE  # 2^32 fragments
    assert decompress_ws(lib, [2**35 - 16]) < NONE
    assert decompress_ws(lib, [2**35 + 1]) == NONE
    assert decompress_ws(lib, [2**35 - 16] * 2) == NONE  # 2 * (2^32 - 1) table entries
    assert lib.csnappy_framed_batch_compress_workspace(None, 3) == NONE


def test_batch_calls_fail_loudly_without_a_device(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: the no-device behaviour cannot be observed")
    buf = C.create_string_buffer(1 << 20)
    p = C.addressof(buf)
    lens, offs = u64([100, 0, 70000]), u64([0, 100, 100])
    ws = compress_ws(lib, lens)
    assert ws < (1 << 20) - 8192
    rc = lib.csnappy_framed_batch_compress(p, offs.ctypes.data, lens.ctypes.data, 3, p, None, 1 << 20, p, 16, p + 8192,
                                           ws, None)
    assert rc == -100  # CSNAPPY_E_DEVICE
    assert b"csnappy_b200" in lib.csnappy_b200_last_error()
    caps = u64([1000, 1000, 1000])
    wsd = decompress_ws(lib, lens)
    rc = lib.csnappy_framed_batch_decompress(p, offs.ctypes.data, lens.ctypes.data, 3, p, offs.ctypes.data,
                                             caps.ctypes.data, p, p, p, p + 8192, wsd, None)
    assert rc == -100
    assert lib.csnappy_framed_batch_decompressed_length(p, offs.ctypes.data, lens.ctypes.data, 3, p, p, None) == -100
    # refused arguments come before any device work
    assert lib.csnappy_framed_batch_compress(p, offs.ctypes.data, lens.ctypes.data, 3, p, None, 1 << 20, p, 8, p, ws,
                                             None) == -101
    assert lib.csnappy_framed_batch_decompress(p, offs.ctypes.data, lens.ctypes.data, 3, p, offs.ctypes.data,
                                               caps.ctypes.data, p, p, p, p, wsd - 1, None) == -101
