"""GPU parity tests (run on the B200 box): the CUDA path, called through the C ABI, against the oracle."""
import bz2
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_img_tif, lf_synth, multiblock_cases

pytestmark = pytest.mark.gpu

G = json.load(open(os.path.join(GOLDEN, "golden.json")))


@pytest.fixture(scope="module")
def L():
    os.environ["LFM_B200_DEBUG_POISON"] = "1"      # poison decode buffers so ordering bugs cannot hide behind stale data
    import lfm_b200
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    lfm_b200.set_devices(0, 1)
    return lfm_b200


def _block_cases():
    rng = np.random.default_rng(11)
    return {
        "poisson18k": rng.poisson(3, 9216).astype(np.uint16).tobytes(),
        "poisson147k": rng.poisson(20, 73728).astype(np.uint16).tobytes(),
        "bright147k": rng.poisson(900, 73728).astype(np.uint16).tobytes(),
        "rand30k": rng.integers(0, 256, 30000, dtype=np.uint8).tobytes(),
        "zeros18432": bytes(18432), "zeros1020": bytes(1020), "const300": np.full(9216, 300, np.uint16).tobytes(),
        "const300_147k": np.full(73728, 300, np.uint16).tobytes(),
        "runs4": np.repeat(rng.integers(0, 256, 5000, dtype=np.uint8), 4).tobytes(),
        "runs255": np.repeat(rng.integers(0, 256, 100, dtype=np.uint8), 255).tobytes(),
        "runs256": np.repeat(rng.integers(0, 256, 100, dtype=np.uint8), 256).tobytes(),
        "abc": b"abc" * 5000, "tiny2": b"\x01\x02", "tiny6": b"aabbaa",
        "sparse": (rng.random(73728) < 0.02).astype(np.uint16).tobytes(),
        "halfzero": np.concatenate([np.zeros(36864, np.uint16), rng.poisson(5, 36864).astype(np.uint16)]).tobytes(),
    }


@pytest.mark.parametrize("name", sorted(_block_cases().keys()))
def test_block_encoder_stage_by_stage(L, oracle, name):
    """every stage of the GPU bzip2 block encoder against the oracle's trace (and the stream against libbz2)"""
    data = _block_cases()[name]
    level = min(9, (len(data) + 99999) // 100000)
    want_stream, blocks = oracle.bz2_compress(data, level, trace=True)
    assert len(blocks) == 1
    b = blocks[0]
    g = L.debug_encode_block(data)
    assert g["nblock"] == b["nblock"], "RLE1 length"
    assert np.array_equal(g["rle1"], b["rle1"]), "RLE1 bytes"
    assert g["crc"] == b["crc"], "block CRC"
    assert g["n_in_use"] == b["n_in_use"]
    assert np.array_equal(g["bwt"], b["bwt"]), "BWT last column"
    assert g["orig_ptr"] == b["orig_ptr"], "origPtr"
    assert g["n_mtf"] == b["n_mtf"] and np.array_equal(g["mtfv"], b["mtfv"]), "MTF/RLE2 symbols"
    assert g["n_groups"] == b["n_groups"] and g["n_sel"] == b["n_sel"]
    assert g["stream"] == want_stream, "bit stream"
    assert g["stream"] == bz2.compress(data, level)


STACKS = {"img_tif": lambda: golden_img_tif(), "synth_40x70x90_n15": lambda: lf_synth((40, 70, 90), 15),
          "synth_1x200x230_n13": lambda: lf_synth((1, 200, 230), 13), "synth_9x64x64_n11": lambda: lf_synth((9, 64, 64), 11)}
_cache = {}


def stack(name):
    if name not in _cache:
        _cache[name] = STACKS[name]()
    return _cache[name]


@pytest.mark.parametrize("idx", range(len(G["files"])))
def test_file_equals_reference_golden(L, tmp_path, idx):
    """.lfm files written through the C ABI are byte-identical to what the UNMODIFIED reference wrote (golden md5s)"""
    e = G["files"][idx]
    a = stack(e["stack"])
    fn = str(tmp_path / "g.lfm")
    L.write_stack(a, fn, header_version=e["hv_in"], nnum=e["nnum"], way=e["way"])
    data = open(fn, "rb").read()
    assert data[0] == e["hv_stored"], "stored predictor / video bit"
    assert len(data) == e["size"] and hashlib.md5(data).hexdigest() == e["md5"]
    back = L.read_stack(fn, way=e["way"])
    assert np.array_equal(back, a), "round trip"


def test_selection_entropies_close_to_reference(L):
    for e in G["entropy"]:
        f0 = np.ascontiguousarray(stack(e["stack"])[e["frame"]])[None]
        L.compress_to_bytes(f0, header_version=0, nnum=e["nnum"], way=e["way"])
        st = L.stats()
        assert st.selected == 1
        got = list(st.entropy)
        for k in range(8):
            # the golden values were summed sequentially in fp32 (thrust stand-in on the CPU); a GPU tree sum differs in the 4th digit
            assert abs(got[k] - e["e"][k]) <= 3e-4 * max(1.0, abs(e["e"][k])), (e["stack"], e["way"], k, got[k], e["e"][k])
        want = max(range(8), key=lambda k: (-e["e"][k], k))
        assert st.predictor == want


def test_oracle_cross_check_on_fresh_data(L, oracle, tmp_path):
    """inputs the goldens never saw: file bytes == oracle file bytes, for every way and a few predictors"""
    rng = np.random.default_rng(99)
    a = (lf_synth((5, 131, 157), 13, seed=4).astype(np.int64) + rng.integers(0, 40, (5, 131, 157))).astype(np.uint16)
    for way in range(3):
        for hv in (0, 8, 9, 12, 15) + ((0x80, 0x8C) if way == 0 else ()):
            fo, fg = str(tmp_path / "o.lfm"), str(tmp_path / "g.lfm")
            rc, shv = oracle.write(a, fo, hv, 13, way, block_size=(64, 48, 4, 1, 1))
            assert rc == 0
            L.write_stack(a, fg, header_version=hv, nnum=13, block_size=(64, 48, 4, 1, 1), way=way)
            assert open(fo, "rb").read() == open(fg, "rb").read(), (way, hex(hv))
            assert np.array_equal(L.read_stack(fg, way=way), a)


@pytest.mark.parametrize("way", [0, 1, 2])
def test_vector_width_frames_all_predictors(L, oracle, tmp_path, way):
    """row length a multiple of 8 pixels (the two-pixels-per-thread forward kernel and the vectorised inverse strips):
    every predictor of every way, file bytes == oracle file bytes, exact round trip"""
    rng = np.random.default_rng(5 + way)
    nz = 18 if way == 0 else 2          # way tiles: enough frames for the one-CTA-per-frame inverse, video halves included
    a = (lf_synth((nz, 120, 272), 13, seed=9).astype(np.int64) + rng.integers(0, 300, (nz, 120, 272))).astype(np.uint16)
    for k in range(1, 8):
        for hv in (8 + k,) + ((0x88 + k,) if way == 0 else ()):
            fo, fg = str(tmp_path / "o.lfm"), str(tmp_path / "g.lfm")
            rc, shv = oracle.write(a, fo, hv, 13, way, block_size=(96, 96, 2, 1, 1))
            assert rc == 0
            L.write_stack(a, fg, header_version=hv, nnum=13, block_size=(96, 96, 2, 1, 1), way=way)
            assert open(fo, "rb").read() == open(fg, "rb").read(), (way, hex(hv))
            assert np.array_equal(L.read_stack(fg, way=way), a)


def test_large_klb_blocks_single_bzip2_block(L, oracle, tmp_path):
    """128x128x6 KLB blocks (196608 bytes, bzip2 level 2: one of the block shapes timed in docs/CompressionComparison.xlsx):
    the text no longer fits shared memory in the block sort, and a block only fits ONE bzip2 block when its run-length
    coded size stays below 100000*level-19 -- checked per block at run time"""
    a = lf_synth((6, 256, 256), 13, seed=21)
    fo, fg = str(tmp_path / "o.lfm"), str(tmp_path / "g.lfm")
    rc, shv = oracle.write(a, fo, 8 + 4, 13, 0, block_size=(128, 128, 6, 1, 1))
    assert rc == 0
    L.write_stack(a, fg, header_version=8 + 4, nnum=13, block_size=(128, 128, 6, 1, 1), way=0)
    assert open(fo, "rb").read() == open(fg, "rb").read()
    assert np.array_equal(L.read_stack(fg, way=0), a)
    # runs of exactly four equal bytes grow by 25 % under bzip2's first run-length stage: 245760 > 199981 -> two bzip2 blocks per stream
    b = np.repeat(np.arange(6 * 256 * 256 // 2, dtype=np.uint32) % 251 * 257, 2).astype(np.uint16).reshape(6, 256, 256)
    rc, shv = oracle.write(b, fo, 8, 13, 0, block_size=(128, 128, 6, 1, 1))
    assert rc == 0
    L.write_stack(b, fg, header_version=8, nnum=13, block_size=(128, 128, 6, 1, 1), way=0)
    assert open(fo, "rb").read() == open(fg, "rb").read()
    assert np.array_equal(L.read_stack(fg, way=0), b)


@pytest.mark.parametrize("name", sorted(multiblock_cases().keys()))
def test_multi_block_streams(L, oracle, tmp_path, name):
    """one KLB block = one bzip2 stream of SEVERAL bzip2 blocks (block shapes above 100000 * level - 19 run-length coded bytes):
    the stream in the file equals the oracle's / libbz2's for the same bytes and level (src/klb_imageIO.cpp:108, :217), and decodes back"""
    data = multiblock_cases()[name]
    a = np.frombuffer(data, np.uint16).reshape(1, 1, -1)
    level = min(9, (len(data) + 99999) // 100000)
    fn = str(tmp_path / "m.lfm")
    L.write_stack(a, fn, header_version=8, nnum=13, block_size=(a.shape[2], 1, 1, 1, 1), way=0)
    blob = open(fn, "rb").read()
    assert blob[0] == 0                                   # predictor off: the block bytes are the raw pixels
    assert blob[320 + 8:] == oracle.bz2_compress(data, level), "stream differs from the oracle (pinned to BZ2_bzBuffToBuffCompress)"
    if name != "l2_exact_plus1":                          # libbz2's streaming API closes the block before the last byte there (test_oracle_bz2.py)
        assert blob[320 + 8:] == bz2.compress(data, level), "stream differs from libbz2"
    assert bz2.decompress(blob[320 + 8:]) == data
    assert int.from_bytes(blob[320:328], "little") == len(blob) - 328
    assert np.array_equal(L.read_stack(fn, way=0), a)


def test_multi_block_streams_in_a_stack(L, oracle, tmp_path):
    """a stack cut into 160x160x8 blocks (409600 bytes, level 5): mixed one- and two-block streams, border blocks, predictor on"""
    rng = np.random.default_rng(12)
    a = lf_synth((8, 300, 330), 13, seed=5)
    a[:, :150, :170] = np.repeat(rng.integers(0, 60000, (8, 150, 85)), 2, axis=2).astype(np.uint16)    # pixel pairs: 4-byte runs
    for hv, way in ((8, 0), (8 + 4, 0), (8 + 3, 2)):
        fo, fg = str(tmp_path / "o.lfm"), str(tmp_path / "g.lfm")
        rc, shv = oracle.write(a, fo, hv, 13, way, block_size=(160, 160, 8, 1, 1))
        assert rc == 0
        L.write_stack(a, fg, header_version=hv, nnum=13, block_size=(160, 160, 8, 1, 1), way=way)
        assert open(fo, "rb").read() == open(fg, "rb").read(), (hv, way)
        assert np.array_equal(L.read_stack(fg, way=way), a)


def test_c_abi_entry_points(L, tmp_path):
    """the six reference entry points: write, header, full read (malloc'd + in place), ROI read"""
    import ctypes as C
    a = lf_synth((6, 50, 70), 13, seed=3)
    fn = os.fsencode(str(tmp_path / "c.lfm"))
    L.set_way(0)
    xyzct = L._u32x5(70, 50, 6, 1, 1)
    assert L.lib.writeKLBstack(a.ctypes.data, fn, xyzct, 1, -1, None, None, 1, None) == 0
    h = L.read_header(fn)
    assert h["xyzct"] == [70, 50, 6, 1, 1] and h["blockSize"] == [70, 50, 6, 1, 1] and h["Nnum"] == 13 and h["dataType"] == 1
    o = np.empty_like(a); dt = C.c_int()
    assert L.lib.readKLBstackInPlace(fn, o.ctypes.data, C.byref(dt), -1) == 0 and np.array_equal(o, a) and dt.value == 1
    x2 = L._u32x5(); dt2 = C.c_int()
    p = L.lib.readKLBstack(fn, x2, C.byref(dt2), -1, None, None, None, None)
    assert p and np.array_equal(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint16)), a.shape), a)
    L._libc.free(p)
    roi = L.read_roi(fn, (5, 7, 1, 0, 0), (40, 30, 4, 0, 0))
    assert np.array_equal(roi[0, 0], a[1:5, 7:31, 5:41])
    # slices API
    ptrs = (C.c_void_p * 6)(*[a[z].ctypes.data for z in range(6)])
    fn2 = os.fsencode(str(tmp_path / "s.lfm"))
    assert L.lib.writeKLBstackSlices(ptrs, fn2, xyzct, 1, -1, None, None, 1, None) == 0
    assert open(fn, "rb").read() == open(fn2, "rb").read()
    # error codes
    assert L.lib.writeKLBstack(a.ctypes.data, b"/nonexistent_dir/x.lfm", xyzct, 1, -1, None, None, 1, None) == 5
    assert L.lib.writeKLBstack(a.ctypes.data, fn2, xyzct, 0, -1, None, None, 1, None) == 7      # uint8: unsupported
    assert L.lib.readKLBstackInPlace(b"/nonexistent.lfm", o.ctypes.data, C.byref(dt), -1) != 0


def test_roi_without_predictor_decodes_only_needed_blocks(L, tmp_path):
    a = lf_synth((20, 120, 130), 13, seed=8)
    fn = str(tmp_path / "r.lfm")
    L.write_stack(a, fn, header_version=8, block_size=(32, 32, 4, 1, 1), way=0)
    for lb, ub in [((0, 0, 7, 0, 0), (129, 119, 7, 0, 0)), ((40, 0, 0, 0, 0), (40, 119, 19, 0, 0)), ((3, 50, 2, 0, 0), (77, 50, 17, 0, 0)),
                   ((33, 31, 3, 0, 0), (64, 95, 12, 0, 0))]:
        r = L.read_roi(fn, lb, ub)
        assert np.array_equal(r[0, 0], a[lb[2]:ub[2] + 1, lb[1]:ub[1] + 1, lb[0]:ub[0] + 1])
    L.write_stack(a, fn, header_version=0x80 | 12, block_size=(32, 32, 4, 1, 1), way=0)
    r = L.read_roi(fn, (10, 20, 5, 0, 0), (100, 90, 9, 0, 0))
    assert np.array_equal(r[0, 0], a[5:10, 20:91, 10:101])


def test_corrupt_file_is_rejected(L, tmp_path):
    a = lf_synth((4, 64, 64), 13)
    fn = str(tmp_path / "x.lfm")
    L.write_stack(a, fn, header_version=8)
    raw = bytearray(open(fn, "rb").read())
    raw[len(raw) - 200] ^= 0x5A
    open(fn, "wb").write(bytes(raw))
    with pytest.raises(L.LfmError) as ei:
        L.read_stack(fn)
    assert ei.value.code == 2


def test_randomised_bzip2_blocks_decode(L, oracle, tmp_path):
    """files whose block streams carry bzip2's "randomised" bit (only bzip2 <= 0.9.0 wrote them; decompress.c BZ_RAND_*): the oracle's
    test hook writes them (pinned to libbz2 in test_oracle_bz2.py), the GPU decoder reads them -- single- and multi-block streams"""
    a = (lf_synth((9, 100, 130), 13, seed=12)).astype(np.uint16)
    fn = str(tmp_path / "r.lfm")
    for hv, bs in ((8, (64, 48, 4, 1, 1)), (8 + 4, (130, 100, 9, 1, 1)), (8, (130, 100, 9, 1, 1))):
        oracle.set_randomised(True)
        try:
            rc, _ = oracle.write(a, fn, hv, 13, 0, block_size=bs)
        finally:
            oracle.set_randomised(False)
        assert rc == 0
        plain = str(tmp_path / "p.lfm")
        rc, _ = oracle.write(a, plain, hv, 13, 0, block_size=bs)
        assert rc == 0 and open(plain, "rb").read() != open(fn, "rb").read()
        assert np.array_equal(L.read_stack(fn, way=0), a), (hv, bs)


def test_memory_and_device_entry_points(L):
    import ctypes as C
    import torch
    a = lf_synth((3, 200, 210), 15, seed=6)
    blob = L.compress_to_bytes(a, header_version=0, nnum=15, way=2)
    assert np.array_equal(L.decompress_from_bytes(blob, a.shape, way=2), a)
    buf = np.empty(len(blob) + 10, np.uint8); back = np.empty_like(a)
    assert L.compress_into(a, buf, header_version=0, nnum=15, way=2) == len(blob) and bytes(buf[:len(blob)]) == blob
    assert np.array_equal(L.decompress_into(buf, len(blob), back, way=2), a)
    with pytest.raises(L.LfmError) as ei:
        L.compress_into(a, buf[:100], header_version=0, nnum=15, way=2)
    assert ei.value.code == 5
    t = torch.from_numpy(a.astype(np.int16)).cuda()
    xyzct = L._u32x5(210, 200, 3, 1, 1)
    nb = L.lib.lfmNumBlocks(xyzct, None)
    off = np.zeros(nb, np.uint64); shv = C.c_uint8(); dp = C.c_void_p(); pb = C.c_uint64()
    assert L.lib.lfmCompressDevice(t.data_ptr(), xyzct, None, 0, 15, C.byref(shv), off.ctypes.data, nb, C.byref(dp), C.byref(pb)) == 0
    assert off[-1] == pb.value and blob[0] == shv.value
    hdr = 320 + 8 * nb
    assert np.array_equal(np.frombuffer(blob[320:hdr], np.uint64), off)
    out = torch.empty_like(t)
    assert L.lib.lfmDecompressDevice(dp, off.ctypes.data, nb, xyzct, None, shv.value, 15, out.data_ptr()) == 0
    torch.cuda.synchronize()
    assert torch.equal(out, t)


def test_large_frame_round_trip_properties(L):
    """BASELINE config 2 size (2048x2048, Nnum 15, space): ratio sanity, determinism, exact round trip"""
    a = lf_synth((1, 2048, 2048), 15)
    b1 = L.compress_to_bytes(a, header_version=8 + 4, nnum=15, way=2)
    b2 = L.compress_to_bytes(a, header_version=8 + 4, nnum=15, way=2)
    assert b1 == b2
    assert np.array_equal(L.decompress_from_bytes(b1, a.shape, way=2), a)
    nb = 22 * 22
    offs = np.frombuffer(b1[320:320 + 8 * nb], np.uint64)
    assert np.all(np.diff(offs.astype(np.int64)) > 0) and offs[-1] == len(b1) - 320 - 8 * nb
    # each block stream is a valid bzip2 stream that libbz2 itself decodes (checksum of checksums)
    pay = b1[320 + 8 * nb:]
    for i in (0, 1, 200, nb - 1):
        s = pay[int(offs[i - 1]) if i else 0:int(offs[i])]
        assert len(bz2.decompress(s)) in (96 * 96 * 2, 96 * 32 * 2, 32 * 96 * 2, 32 * 32 * 2)


def test_two_gpus_in_process_sharding(L, tmp_path):
    """lfmSetDevices(0, 2): z-slabs split over two GPUs, host prefix sum -> same bytes as one GPU"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    a = lf_synth((24, 100, 120), 13, seed=2)
    one = L.compress_to_bytes(a, header_version=0x80 | 13, nnum=13, block_size=(48, 48, 4, 1, 1), way=0)
    try:
        assert L.set_devices(0, 2) == 2
        two = L.compress_to_bytes(a, header_version=0x80 | 13, nnum=13, block_size=(48, 48, 4, 1, 1), way=0)
        assert one == two
        assert np.array_equal(L.decompress_from_bytes(two, a.shape, way=0), a)
    finally:
        L.set_devices(0, 1)


@pytest.mark.parametrize("shape_t", [((40, 300, 520), 13), ((7, 95, 333), 15), ((160, 64, 200), 5)])
def test_inverse_band_pipeline_many_frames(L, shape_t):
    """way tiles, stacks of >= 3 frames: the band-pipelined inverse (one CTA per band of tile rows, bands of a frame chained
    through progress flags, more bands than fit the GPU at once).  Every predictor, image and video mode: the inverse applied
    to the forward kernel's symbols restores the stack exactly (the forward kernel is pinned to the oracle by the file tests)."""
    import ctypes as C
    import torch
    (F, H, W), T = shape_t
    rng = np.random.default_rng(F)
    a = (lf_synth((F, H, W), T, seed=3).astype(np.int64) + rng.integers(0, 500, (F, H, W))).astype(np.uint16)
    d = torch.from_numpy(a.view(np.int16)).cuda()
    sym = torch.empty_like(d); back = torch.empty_like(d)
    xyz = L._u32x5(W, H, F, 1, 1)
    ms = C.c_float()
    prev = L.set_way(0)
    try:
        for k in range(1, 8):
            for video in (0, 1):
                back.fill_(-21555)
                assert L.lib.lfmDebugPredictDevice(d.data_ptr(), sym.data_ptr(), xyz, T, k, video, 0, 1, C.byref(ms)) == 0
                assert L.lib.lfmDebugPredictDevice(sym.data_ptr(), back.data_ptr(), xyz, T, k, video, 1, 1, C.byref(ms)) == 0
                assert torch.equal(back, d), (k, video)
    finally:
        L.set_way(prev if prev is not None and prev >= 0 else 0)


def test_roi_reads_with_predictors(L, tmp_path):
    """readImage(ROI) (src/klb_imageIO.cpp:2614-2682) on predicted files: only the slabs the ROI touches are fetched from the file
    (byte-range reads) and, inside them, only the KLB blocks up / left of the ROI's lower right corner are decoded -- the
    prediction rules never look right or down -- every way, image and video mode, random boxes, planes and single pixels"""
    rng = np.random.default_rng(31)
    a = (lf_synth((9, 150, 170), 13, seed=8).astype(np.int64) + rng.integers(0, 200, (9, 150, 170))).astype(np.uint16)
    fn = str(tmp_path / "r.lfm")
    for way, hv in ((0, 0), (0, 8 + 7), (0, 0x80 | 12), (0, 8 + 2), (1, 8 + 5), (1, 8 + 2), (2, 0), (2, 8 + 6), (0, 8)):
        L.write_stack(a, fn, header_version=hv, nnum=13, block_size=(32, 32, 4, 1, 1), way=way)
        boxes = [((0, 0, 0), (169, 149, 8)), ((0, 0, 4), (169, 149, 4)), ((169, 149, 8), (169, 149, 8)), ((0, 0, 0), (0, 0, 0)), ((5, 0, 3), (5, 149, 5))]
        for _ in range(6):
            lo = [int(rng.integers(0, n)) for n in (170, 150, 9)]
            hi = [int(rng.integers(lo[i], n)) for i, n in enumerate((170, 150, 9))]
            boxes.append((tuple(lo), tuple(hi)))
        for lo, hi in boxes:
            r = L.read_roi(fn, lo + (0, 0), hi + (0, 0), way=way)
            assert np.array_equal(r[0, 0], a[lo[2]:hi[2] + 1, lo[1]:hi[1] + 1, lo[0]:hi[0] + 1]), (way, hex(hv), lo, hi)


def test_pageable_stacks_take_the_staged_copy_path(L, tmp_path):
    """callers of the reference API pass malloc'ed stacks: copies of >= 16 MB of pageable memory go through the engine's pinned
    staging buffers (klb_imageIO.cpp h2d_staged / d2h_staged).  Same file bytes as with pinned buffers (direct DMA), exact read back."""
    import torch
    a = lf_synth((3, 2048, 2048), 13, seed=17)                       # 25 MB, pageable numpy memory
    fn = str(tmp_path / "p.lfm")
    L.write_stack(a, fn, header_version=8 + 4, nnum=13, way=0)
    hin = torch.from_numpy(a.view(np.int16)).pin_memory()
    blob = torch.empty(a.nbytes, dtype=torch.uint8).pin_memory()
    n = L.compress_into(hin.numpy().view(np.uint16), blob.numpy(), header_version=8 + 4, nnum=13, way=0)
    assert open(fn, "rb").read() == blob.numpy()[:n].tobytes()
    assert np.array_equal(L.read_stack(fn, way=0), a)
    back = np.empty_like(a)
    L.decompress_into(blob.numpy(), n, back, way=0)                  # pinned source, pageable destination
    assert np.array_equal(back, a)


@pytest.mark.parametrize("frames", [3, 9])
def test_inverse_fallback_kernels_large_nnum(L, oracle, frames):
    """Nnum = 33: a tile no longer fits the band pipeline (Nnum^2 threads) nor the column kernel's shuffle chain (Nnum <= 32), and
    the strips kernel's shared memory only holds Nnum <= 22, so the way tiles / angle inverses fall back to the cluster wavefront
    (predictor 2 of those ways: its row schedule).  Every predictor, image and video mode: forward symbols of frame 0 equal the
    oracle's, inverse(forward) restores the stack.  (tests/test_predict_dispatch.py pins the strips kernel.)"""
    import ctypes as C
    import torch
    T, H, W = 33, 100, 136
    rng = np.random.default_rng(frames)
    a = (lf_synth((frames, H, W), T, seed=2).astype(np.int64) + rng.integers(0, 300, (frames, H, W))).astype(np.uint16)
    d = torch.from_numpy(a.view(np.int16)).cuda()
    sym = torch.empty_like(d); back = torch.empty_like(d)
    xyz = L._u32x5(W, H, frames, 1, 1)
    ms = C.c_float()
    prev = L.set_way(0)
    try:
        for way in (0, 1, 2):
            L.set_way(way)
            for k in range(1, 8):
                for video in ((0, 1) if way == 0 else (0,)):
                    back.fill_(-21555)
                    assert L.lib.lfmDebugPredictDevice(d.data_ptr(), sym.data_ptr(), xyz, T, k, video, 0, 1, C.byref(ms)) == 0
                    want0 = oracle.predict_frame(a[0], None, T, way, k, 0)
                    assert np.array_equal(sym[0].cpu().numpy().view(np.uint16), want0), (way, k, video)
                    assert L.lib.lfmDebugPredictDevice(sym.data_ptr(), back.data_ptr(), xyz, T, k, video, 1, 1, C.byref(ms)) == 0
                    assert torch.equal(back, d), (way, k, video)
    finally:
        L.set_way(prev if prev is not None and prev >= 0 else 0)
