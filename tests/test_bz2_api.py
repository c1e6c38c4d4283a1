"""Standalone bzip2 streams (lfmBz2Compress / lfmBz2CompressDevice, bz2_compress): byte parity with BZ2_bzBuffToBuffCompress."""
import bz2
import ctypes as C
import importlib

import numpy as np
import pytest

from conftest import has_cuda, lf_synth, multiblock_cases
from test_oracle_bz2 import STREAMING_DIFFERS, _cases, _vendored_bz2

M1 = 99981                       # nblockMAX at level 1: run-length coded bytes that close a block


@pytest.fixture(scope="module")
def L():
    return importlib.import_module("lightfieldmicroscopy_pc-bzip2_b200")


def _norun(rng, n):
    """bytes without two equal neighbours: every byte is a record of its own"""
    a = rng.integers(0, 255, n, dtype=np.uint8)
    a[1:] += (a[1:] >= a[:-1]).astype(np.uint8)          # a[i] != a[i-1] except where the shift lands on it again
    for i in np.nonzero(a[1:] == a[:-1])[0]:
        a[i + 1] = (int(a[i]) + 7) % 256
    return a


def _runs300_across_limits(seed=9, blocks=12):
    """literal filler with a 300-byte run starting 0..9 output bytes before each of the first `blocks` level-1 block limits
    (a 300-run is two records, 255 + 45, ten output bytes)"""
    rng = np.random.default_rng(seed)
    parts, out_pos = [], 0
    for k in range(1, blocks + 1):
        start = k * M1 - (k * 7) % 10
        f = _norun(rng, start - out_pos)
        v = (int(f[-1]) + 1) % 256
        parts += [f, np.full(300, v, np.uint8), np.array([(v + 1) % 256], np.uint8)]
        out_pos = start + 10 + 1
    parts.append(_norun(rng, 5000))
    return np.concatenate(parts).tobytes()


def _check_parity(L, oracle, data, level, name, ref=None):
    got = L.bz2_compress(data, level)
    want = oracle.bz2_compress(data, level)
    assert got == want, (name, level, len(got), len(want))
    if ref is not None:
        assert got == ref(data, level), (name, level, "libbz2 BZ2_bzBuffToBuffCompress")
    if not (name in STREAMING_DIFFERS and level == 2):
        assert got == bz2.compress(data, level), (name, level, "bz2.compress")
    return got


# ---------------------------------------------------------------------------------------------------- no GPU needed
def test_bz2_entry_points_exported(L):
    for name in ("lfmBz2Compress", "lfmBz2CompressDevice"):
        assert name in L.EXPORTS and hasattr(L.lib, name)


@pytest.mark.parametrize("level", [0, 10, -1])
def test_bz2_bad_level_is_rejected_before_any_device_work(L, level):
    n = C.c_uint64(123)
    buf = (C.c_uint8 * 64)()
    assert L.lib.lfmBz2Compress(b"abc", 3, level, buf, 64, C.byref(n)) == 3
    p = C.c_void_p()
    assert L.lib.lfmBz2CompressDevice(None, 0, level, C.byref(p), C.byref(n)) == 3


def test_bz2_null_input_with_bytes_is_rejected(L):
    n = C.c_uint64()
    buf = (C.c_uint8 * 64)()
    assert L.lib.lfmBz2Compress(None, 5, 9, buf, 64, C.byref(n)) == 3
    p = C.c_void_p()
    assert L.lib.lfmBz2CompressDevice(None, 5, 9, C.byref(p), C.byref(n)) == 3


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 2, 5, 9])
def test_bz2_compress_matches_libbz2_oracle_cases(L, oracle, level):
    ref = _vendored_bz2()
    for name, data in _cases().items():
        _check_parity(L, oracle, data, level, name, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("level", [1, 2, 5, 9])
def test_bz2_compress_matches_libbz2_multiblock_cases(L, oracle, level):
    ref = _vendored_bz2()
    for name, data in multiblock_cases().items():
        _check_parity(L, oracle, data, level, name, ref)


@pytest.mark.gpu
def test_bz2_compress_small_and_odd_lengths(L, oracle):
    rng = np.random.default_rng(4)
    for n in (0, 1, 2, 3, 17, 255, 1001, 4097, 8191, 8193, 99983):
        for data in (rng.integers(0, 256, n, dtype=np.uint8).tobytes(), bytes(n), np.repeat(rng.integers(0, 3, n), 1)[:n].astype(np.uint8).tobytes()):
            for level in (1, 9):
                _check_parity(L, oracle, data, level, "len%d" % n)
    assert L.bz2_compress(b"", 9) == bz2.compress(b"", 9) and len(L.bz2_compress(b"", 9)) == 14


@pytest.mark.gpu
def test_bz2_compress_runs_across_block_limits(L, oracle):
    data = _runs300_across_limits()
    _check_parity(L, oracle, data, 1, "runs300", _vendored_bz2())
    assert len(oracle.bz2_compress(data, 1, trace=True)[1]) == 13
    # and the same idea with runs that tile-borders of the run-length pass cut (long runs, every length mod 255)
    rng = np.random.default_rng(10)
    lens = rng.choice([1, 2, 3, 4, 5, 254, 255, 256, 259, 300, 510, 9000, 20000], 3000)
    vals = _norun(rng, len(lens))
    data = np.repeat(vals, lens).tobytes()
    for level in (1, 2):
        _check_parity(L, oracle, data, level, "mixed_runs")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["lf_synth", "random"])
def test_bz2_compress_20mb_streams(L, oracle, kind):
    if kind == "lf_synth":
        data = lf_synth((5, 1024, 2048), 13, seed=21).tobytes()      # 20 MiB of uint16 pixels
    else:
        data = np.random.default_rng(22).integers(0, 256, 20 << 20, dtype=np.uint8).tobytes()
    for level in (1, 9):
        got = _check_parity(L, oracle, data, level, kind)
        st = L.stats()
        assert st.payload_bytes == len(got) and st.gpu_launches > 0
        assert st.ms_rle > 0 and st.ms_bwt > 0 and st.ms_mtf > 0 and st.ms_huff > 0


@pytest.mark.gpu
def test_bz2_compress_accepts_numpy_and_memoryview(L):
    a = np.arange(40000, dtype=np.uint16) % 300
    want = bz2.compress(a.tobytes(), 5)
    assert L.bz2_compress(a, 5) == want
    assert L.bz2_compress(memoryview(a.tobytes()), 5) == want
    assert L.bz2_compress(bytearray(a.tobytes()), 5) == want


@pytest.mark.gpu
def test_bz2_rejections(L):
    data = np.random.default_rng(6).integers(0, 256, 300000, dtype=np.uint8).tobytes()
    for level in (0, 10):
        with pytest.raises(L.LfmError) as e:
            L.bz2_compress(data, level)
        assert e.value.code == 3
    need = len(bz2.compress(data, 3))
    guard = 16
    buf = (C.c_uint8 * (need + guard))(*([0xA5] * (need + guard)))
    n = C.c_uint64(0)
    assert L.lib.lfmBz2Compress(data, len(data), 3, buf, need - 1, C.byref(n)) == 5
    assert n.value == need
    assert bytes(buf) == b"\xa5" * (need + guard)                  # nothing written, not even the guard bytes after dst
    assert L.lib.lfmBz2Compress(data, len(data), 3, buf, need, C.byref(n)) == 0
    assert bytes(buf)[:need] == bz2.compress(data, 3) and bytes(buf)[need:] == b"\xa5" * guard


@pytest.mark.gpu
def test_bz2_device_and_host_agree(L):
    import torch
    if not has_cuda():
        pytest.skip("no CUDA device")
    rng = np.random.default_rng(8)
    for data in (b"", b"z", lf_synth((2, 300, 700), 13, seed=3).tobytes(), rng.integers(0, 256, 1500000, dtype=np.uint8).tobytes()):
        t = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda() if data else torch.empty(0, dtype=torch.uint8, device="cuda")
        for level in (1, 9):
            d = L.bz2_compress(t, level)
            assert d.is_cuda and d.dtype == torch.uint8
            assert bytes(d.cpu().numpy()) == L.bz2_compress(data, level) == bz2.compress(data, level)
    # a view into a larger tensor (odd byte offset) and a non-uint8 tensor
    big = torch.frombuffer(bytearray(rng.integers(0, 256, 70001, dtype=np.uint8).tobytes()), dtype=torch.uint8).cuda()
    assert bytes(L.bz2_compress(big[3:], 2).cpu().numpy()) == bz2.compress(bytes(big[3:].cpu().numpy()), 2)
    with pytest.raises(TypeError):
        L.bz2_compress(big.to(torch.int16), 9)


@pytest.mark.gpu
def test_bz2_calls_leave_the_klb_path_unchanged(L):
    img = lf_synth((6, 260, 390), 13, seed=31)
    file0 = L.compress_to_bytes(img, header_version=8 + 3)
    back0 = L.decompress_from_bytes(file0, img.shape)
    L.bz2_compress(np.random.default_rng(1).integers(0, 256, 3000000, dtype=np.uint8).tobytes(), 9)
    L.bz2_compress(bytes(100), 1)
    file1 = L.compress_to_bytes(img, header_version=8 + 3)
    back1 = L.decompress_from_bytes(file1, img.shape)
    assert file1 == file0
    assert np.array_equal(back1, back0) and np.array_equal(back1, img)
