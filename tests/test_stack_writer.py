"""Recording a stack frame by frame (StackWriter; lfmStackWriterOpen / Append / AppendDevice / Close in include/lfm_b200.h).
A recording closed with every declared frame must be byte-identical to write_stack of the whole stack, whatever the append chunking
and whether the frames came from host or device memory; one closed early must be byte-identical to write_stack of the kept prefix.
write_stack of a large stack goes through the same writer, so the references are written with LFM_B200_NO_PIPELINE=1: by the
one-shot path, which compresses the stack in one pass without the writer (a stack writer always batches)."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from conftest import has_cuda, lf_synth, lf_synth_int


@pytest.fixture(scope="module")
def L():
    import lfm_b200
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    lfm_b200.set_devices(0, 1)
    return lfm_b200


@pytest.fixture(scope="module")
def Lhost():
    import lfm_b200
    return lfm_b200


def _md5(fn):
    return hashlib.md5(open(fn, "rb").read()).hexdigest()


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda()


def _frames(a):
    """[t][c][z][y][x] or [z][y][x] -> [frames][y][x] in arrival order"""
    return a.reshape(-1, a.shape[-2], a.shape[-1])


def _pair_runs(shape, seed):
    """lf_synth with a corner of pixel pairs (4-byte runs): cut into 160x160x8 blocks, some streams hold two bzip2 blocks"""
    rng = np.random.default_rng(12)
    a = lf_synth(shape, 13, seed=seed)
    a[:, :150, :170] = np.repeat(rng.integers(0, 60000, (shape[0], 150, 85)), 2, axis=2).astype(np.uint16)
    return a


# name: (stack, write_stack keyword arguments, LFM_B200_BATCH_KB or None) -- the kinds of stacks test_device_io.py writes
def _cases():
    c = {}
    for way in (0, 1, 2):
        for hv in (0, 8, 8 + 4, 8 + 7):
            c["way%d_hv%d" % (way, hv)] = (lambda: lf_synth((9, 150, 170), 13, seed=8),
                                           dict(header_version=hv, block_size=(64, 64, 4, 1, 1), way=way), None)
    for hv in (0x80, 0x80 | 12):
        c["video_%x_odd_depth" % hv] = (lambda: lf_synth((10, 100, 120), 13, seed=4),
                                        dict(header_version=hv, block_size=(64, 64, 3, 1, 1), way=0), None)
    c["multi_block_streams"] = (lambda: _pair_runs((8, 300, 330), 5), dict(header_version=8 + 4, block_size=(160, 160, 8, 1, 1), way=0), None)
    c["channels_times"] = (lambda: lf_synth((30, 60, 70), 13, seed=3).reshape(2, 3, 5, 60, 70),
                           dict(header_version=8 + 4, block_size=(32, 32, 2, 1, 1), way=0), None)
    c["codec_none"] = (lambda: lf_synth((7, 150, 170), 13, seed=9), dict(header_version=8 + 5, block_size=(64, 48, 4, 1, 1), way=0, codec=0), None)
    c["slab_pipeline_auto"] = (lambda: lf_synth((45, 200, 230), 13, seed=11), dict(header_version=0, block_size=(64, 64, 4, 1, 1), way=0), 400)
    c["slab_pipeline_video"] = (lambda: lf_synth((45, 200, 230), 13, seed=11), dict(header_version=0x80 | 12, block_size=(64, 64, 3, 1, 1), way=0), 300)
    c["slab_pipeline_raw"] = (lambda: lf_synth((45, 200, 230), 13, seed=11), dict(header_version=8, block_size=(96, 96, 1, 1, 1), way=0), 100)
    # video volumes whose depth is not a multiple of the block depth: slabs in the middle start on odd frames (5 = 2 + 2 + 1: the
    # slabs of volume 1 start at frames 5, 7, 9), and a batch must still start on an even one
    c["video_volumes_z5_t8"] = (lambda: lf_synth((40, 100, 120), 13, seed=14).reshape(8, 1, 5, 100, 120),
                                dict(header_version=0x80 | 12, block_size=(64, 64, 2, 1, 1), way=0), 60)
    c["video_volumes_z7_t3_auto"] = (lambda: lf_synth((21, 100, 120), 13, seed=15).reshape(3, 1, 7, 100, 120),
                                     dict(header_version=0x80, block_size=(64, 64, 2, 1, 1), way=0), 100)
    c["video_volumes_z5_c2_t3_odd_depth"] = (lambda: lf_synth((30, 100, 120), 13, seed=16).reshape(3, 2, 5, 100, 120),
                                             dict(header_version=0x80 | 9, block_size=(64, 64, 3, 1, 1), way=0), 70)
    return c


CASES = _cases()


def _chunks(n, how, seed):
    if how == "one":
        return [1] * n
    if how == "whole":
        return [n]
    rng = np.random.default_rng(seed)
    out = []
    while sum(out) < n:
        out.append(int(min(n - sum(out), rng.integers(1, 8))))
    return out


def _record(L, fn, a, kw, chunks, source, nframes=None):
    """append the first `nframes` frames of `a` in `chunks` from `source` (numpy, cuda or alternating); returns close()"""
    fr = _frames(a)
    dev = _cuda(fr) if source != "numpy" else None
    w = L.StackWriter(fn, a.shape, nnum=13, **kw)
    f = 0
    for i, n in enumerate(chunks):
        if nframes is not None:
            n = min(n, nframes - f)
        if n <= 0:
            break
        on_dev = source == "cuda" or (source == "alternate" and i % 2 == 1)
        part = dev[f:f + n] if on_dev else fr[f:f + n]
        w.append(part[0] if n == 1 and i % 3 == 0 else part)          # [y][x] as well as [n][y][x]
        f += n
    return w.close()


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["numpy", "cuda", "alternate"])
@pytest.mark.parametrize("chunking", ["one", "random", "whole"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_recording_is_byte_identical_to_write_stack(L, tmp_path, monkeypatch, name, chunking, source):
    make, kw, batch_kb = CASES[name]
    if batch_kb:
        monkeypatch.setenv("LFM_B200_BATCH_KB", str(batch_kb))          # batches of a few slabs
    monkeypatch.setenv("LFM_B200_NO_PIPELINE", "1")                      # the reference: the one-shot path
    a = make()
    ref, rec = str(tmp_path / "ref.lfm"), str(tmp_path / "rec.lfm")
    L.write_stack(a, ref, nnum=13, **kw)
    n = _frames(a).shape[0]
    assert _record(L, rec, a, kw, _chunks(n, chunking, seed=len(name)), source) == n
    assert _md5(rec) == _md5(ref), (name, chunking, source)
    assert np.array_equal(L.read_stack(rec, way=kw["way"]), a)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_write_stack_through_the_writer_matches_the_one_shot_path(L, tmp_path, monkeypatch, name):
    """write_stack of a stack of two batches or more goes through the writer: same file as the one-shot path, and the batched
    read (host and device output) returns the pixels"""
    import torch
    make, kw, batch_kb = CASES[name]
    if batch_kb:
        monkeypatch.setenv("LFM_B200_BATCH_KB", str(batch_kb))
    a = make()
    one, piped = str(tmp_path / "one.lfm"), str(tmp_path / "piped.lfm")
    monkeypatch.setenv("LFM_B200_NO_PIPELINE", "1")
    L.write_stack(a, one, nnum=13, **kw)
    monkeypatch.delenv("LFM_B200_NO_PIPELINE")
    L.write_stack(a, piped, nnum=13, **kw)
    assert _md5(piped) == _md5(one), name
    assert np.array_equal(L.read_stack(piped, way=kw["way"]), a)
    assert torch.equal(L.read_stack(piped, way=kw["way"], device="cuda").view(torch.int16), _cuda(a))


@pytest.mark.gpu
def test_video_volumes_at_the_default_batch_size(L, tmp_path, monkeypatch):
    """2048^2 frames, 7-frame volumes, 96x96x2 blocks, video bit + predictor 4, no batch knob: 6 slabs per batch would start batch 1
    on frame 11; the batches start on even frames, and the recording, write_stack and the one-shot path give one file"""
    import torch
    d = lf_synth_int((21, 2048, 2048), 13, seed=9, device="cuda")
    a = d.cpu().numpy().view(np.uint16).reshape(3, 1, 7, 2048, 2048)
    kw = dict(header_version=0x80 | 12, block_size=(96, 96, 2, 1, 1), way=0)
    one, piped, rec = str(tmp_path / "one.lfm"), str(tmp_path / "piped.lfm"), str(tmp_path / "rec.lfm")
    monkeypatch.setenv("LFM_B200_NO_PIPELINE", "1")
    L.write_stack(a, one, nnum=13, **kw)
    monkeypatch.delenv("LFM_B200_NO_PIPELINE")
    L.write_stack(a, piped, nnum=13, **kw)
    assert _md5(piped) == _md5(one)
    w = L.StackWriter(rec, a.shape, nnum=13, **kw)
    for f in range(21):
        w.append(d[f] if f % 2 else a.reshape(21, 2048, 2048)[f])
    assert w.close() == 21
    assert _md5(rec) == _md5(one)
    assert np.array_equal(L.read_stack(rec, way=0), a)
    assert torch.equal(L.read_stack(rec, way=0, device="cuda").view(torch.int16).reshape(21, 2048, 2048), d)


@pytest.mark.gpu
def test_recording_stats_are_the_totals(L, tmp_path, monkeypatch):
    monkeypatch.setenv("LFM_B200_BATCH_KB", "400")
    a = lf_synth((45, 200, 230), 13, seed=11)
    kw = dict(header_version=0, block_size=(64, 64, 4, 1, 1), way=0)
    L.write_stack(a, str(tmp_path / "ref.lfm"), nnum=13, **kw)
    want = L.stats()
    _record(L, str(tmp_path / "rec.lfm"), a, kw, [1] * 45, "numpy")
    got = L.stats()
    assert got.selected == 1 and got.predictor == want.predictor
    assert list(got.entropy) == list(want.entropy)
    assert got.payload_bytes == want.payload_bytes == os.path.getsize(str(tmp_path / "rec.lfm")) - 320 - 8 * L.lib.lfmNumBlocks(L._xyzct(a.shape), C.cast(L._bs(kw["block_size"]), C.c_void_p))
    assert got.ms_bwt > 0 and got.ms_huff > 0 and got.gpu_launches >= want.gpu_launches


# ---- early close: (stack, keyword arguments, LFM_B200_BATCH_KB, frames appended, frames kept)
EARLY = {
    "z_mid_block": (lambda: lf_synth((20, 150, 170), 13, seed=1), dict(header_version=8 + 4, block_size=(64, 64, 8, 1, 1), way=0), 400, 13, 13),
    "z_mid_block_auto": (lambda: lf_synth((20, 150, 170), 13, seed=1), dict(header_version=0, block_size=(64, 64, 8, 1, 1), way=1), None, 11, 11),
    "z_less_than_one_block": (lambda: lf_synth((20, 150, 170), 13, seed=1), dict(header_version=8 + 4, block_size=(64, 64, 8, 1, 1), way=0), 400, 5, 5),
    "t_cut_partial_volume": (lambda: lf_synth((24, 100, 120), 13, seed=2).reshape(4, 2, 3, 100, 120),
                             dict(header_version=8 + 4, block_size=(64, 64, 2, 1, 1), way=2), 150, 16, 12),
    "c_cut": (lambda: lf_synth((15, 100, 120), 13, seed=2).reshape(1, 3, 5, 100, 120),
              dict(header_version=8 + 2, block_size=(64, 64, 2, 1, 1), way=0), 60, 13, 10),
    "video_odd_frame": (lambda: lf_synth((11, 100, 120), 13, seed=4), dict(header_version=0x80 | 12, block_size=(64, 64, 3, 1, 1), way=0), 60, 7, 7),
    "video_auto_odd_frame": (lambda: lf_synth((11, 100, 120), 13, seed=4), dict(header_version=0x80, block_size=(64, 64, 3, 1, 1), way=0), None, 9, 9),
    "video_volumes_t_cut": (lambda: lf_synth((40, 100, 120), 13, seed=14).reshape(8, 1, 5, 100, 120),
                            dict(header_version=0x80 | 12, block_size=(64, 64, 2, 1, 1), way=0), 60, 23, 20),
}


def _prefix(a, kept):
    if a.ndim == 3:
        return a[:kept]
    t, c, z = a.shape[:3]
    if t > 1:
        return a[:kept // (c * z)]
    return a[:, :kept // z]


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["numpy", "cuda"])
@pytest.mark.parametrize("name", sorted(EARLY))
def test_early_close_keeps_the_prefix(L, tmp_path, monkeypatch, name, source):
    make, kw, batch_kb, appended, kept = EARLY[name]
    if batch_kb:
        monkeypatch.setenv("LFM_B200_BATCH_KB", str(batch_kb))
    monkeypatch.setenv("LFM_B200_NO_PIPELINE", "1")                      # the reference: the one-shot path
    a = make()
    rec, ref = str(tmp_path / "rec.lfm"), str(tmp_path / "ref.lfm")
    assert _record(L, rec, a, kw, [1] * appended, source) == kept
    p = _prefix(a, kept)
    L.write_stack(p, ref, nnum=13, **kw)
    assert _md5(rec) == _md5(ref), name
    assert np.array_equal(L.read_stack(rec, way=kw["way"]), p)


@pytest.mark.gpu
def test_nothing_kept_is_code_2_and_an_empty_file(L, tmp_path):
    a = lf_synth((18, 100, 120), 13, seed=2).reshape(3, 2, 3, 100, 120)
    for appended in (0, 4):
        fn = str(tmp_path / ("rec%d.lfm" % appended))
        w = L.StackWriter(fn, a.shape, header_version=8 + 4, nnum=13, block_size=(64, 64, 2, 1, 1), way=0)
        if appended:
            w.append(_frames(a)[:appended])
        with pytest.raises(L.LfmError) as ei:
            w.close()
        assert ei.value.code == 2
        assert os.path.getsize(fn) == 0


# ---- errors
def _open(L, fn, shape, dtype=1, codec=1, hv=0, block_size=None):
    w = C.c_void_p()
    bs = L._bs(block_size)
    rc = L.lib.lfmStackWriterOpen(C.byref(w), fn, L._xyzct(shape), dtype, None, C.cast(bs, C.c_void_p) if bs is not None else None,
                                  codec, None, hv, 13)
    return rc, w


@pytest.mark.gpu
def test_open_errors_match_write_stack(L, tmp_path):
    a = lf_synth((4, 60, 70), 13, seed=5)
    cases = [  # (name, dtype, codec, hv, way, filename)
        ("uint8 pixels", 0, 1, 0, 0, None), ("float pixels", 9, 1, 0, 0, None), ("zlib", 1, 2, 0, 0, None),
        ("video forced way 1", 1, 1, 0x80 | 12, 1, None), ("video forced way 2", 1, 1, 0x80 | 9, 2, None),
        ("empty filename", 1, 1, 0, 0, b""), ("no directory", 1, 1, 0, 0, b"/nonexistent_dir/x.lfm"),
    ]
    for i, (what, dtype, codec, hv, way, fname) in enumerate(cases):
        L.set_way(way)
        fw = fname if fname is not None else os.fsencode(str(tmp_path / ("w%d.lfm" % i)))
        fx = fname if fname is not None else os.fsencode(str(tmp_path / ("x%d.lfm" % i)))
        want = L.lib.writeLFMstackEx(a.ctypes.data, fx, L._xyzct(a.shape), dtype, -1, None, None, codec, None, hv, 13)
        rc, w = _open(L, fw, a.shape, dtype, codec, hv)
        assert rc == want != 0 and not w.value, what
        if fw:
            assert not os.path.exists(fw), what
    L.set_way(0)
    fw = str(tmp_path / "blocked.lfm")
    for bs in ((32, 32, 2, 2, 1), (32, 32, 2, 1, 2)):
        rc, w = _open(L, os.fsencode(fw), (2, 3, 5, 60, 70), block_size=bs)
        assert rc == 7 and not os.path.exists(fw)


@pytest.mark.gpu
def test_over_append_keeps_the_writer_usable(L, tmp_path, monkeypatch):
    a = lf_synth((5, 100, 120), 13, seed=6)
    kw = dict(header_version=8 + 3, block_size=(64, 64, 2, 1, 1), way=0)
    rec, ref = str(tmp_path / "rec.lfm"), str(tmp_path / "ref.lfm")
    with L.StackWriter(rec, a.shape, nnum=13, **kw) as w:
        w.append(a[:3])
        with pytest.raises(L.LfmError) as ei:
            w.append(a[:3])
        assert ei.value.code == 3
        w.append(_cuda(a[3:]))
        with pytest.raises(L.LfmError) as ei:
            w.append(a[:1])
        assert ei.value.code == 3
    L.write_stack(a, ref, nnum=13, **kw)
    assert _md5(rec) == _md5(ref)


@pytest.mark.gpu
def test_failed_writer_returns_its_code_and_leaves_an_empty_file(L, tmp_path):
    """auto-selection on a video stack with way 1: writeLFMstackEx refuses with 7 once the predictor is picked, the writer on the
    append that carries frame 0; later appends and Close return the same code and the file is cut to 0 bytes"""
    a = lf_synth((6, 100, 120), 13, seed=7)
    kw = dict(header_version=0x80, block_size=(64, 64, 2, 1, 1), way=1)
    with pytest.raises(L.LfmError) as ei:
        L.write_stack(a, str(tmp_path / "ref.lfm"), nnum=13, **kw)
    assert ei.value.code == 7
    rec = str(tmp_path / "rec.lfm")
    w = L.StackWriter(rec, a.shape, nnum=13, **kw)
    for part in (a[:2], a[2:3]):
        with pytest.raises(L.LfmError) as ei:
            w.append(part)
        assert ei.value.code == 7
    with pytest.raises(L.LfmError) as ei:
        w.close()
    assert ei.value.code == 7 and os.path.getsize(rec) == 0
    # an exception inside the with block is the one raised; the writer is closed all the same
    rec2 = str(tmp_path / "rec2.lfm")
    with pytest.raises(ZeroDivisionError):
        with L.StackWriter(rec2, a.shape, nnum=13, header_version=8 + 4, block_size=(64, 64, 2, 1, 1), way=0) as w2:
            w2.append(a[:4])
            1 / 0
    assert w2.close() == 4
    L.write_stack(a[:4], str(tmp_path / "ref4.lfm"), nnum=13, header_version=8 + 4, block_size=(64, 64, 2, 1, 1), way=0)
    assert _md5(rec2) == _md5(str(tmp_path / "ref4.lfm"))


@pytest.mark.gpu
def test_tensor_on_another_device_is_refused(L, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    a = lf_synth((4, 60, 70), 13, seed=5)
    rec = str(tmp_path / "rec.lfm")
    w = L.StackWriter(rec, a.shape, nnum=13, header_version=8 + 4, way=0)
    with pytest.raises(L.LfmError) as ei:
        w.append(_cuda(a).to("cuda:1"))
    assert ei.value.code == 3
    with pytest.raises(L.LfmError) as ei:
        w.close()
    assert ei.value.code == 3 and os.path.getsize(rec) == 0


# ---- coexistence
@pytest.mark.gpu
def test_two_writers_and_other_calls_between_appends(L, tmp_path, monkeypatch):
    import torch
    monkeypatch.setenv("LFM_B200_BATCH_KB", "300")
    a = lf_synth((45, 200, 230), 13, seed=11)
    b = lf_synth((30, 150, 170), 13, seed=12)
    kwa = dict(header_version=0, block_size=(64, 64, 4, 1, 1), way=0)
    kwb = dict(header_version=0x80 | 12, block_size=(64, 64, 3, 1, 1), way=0)
    refa, refb, other = str(tmp_path / "refa.lfm"), str(tmp_path / "refb.lfm"), str(tmp_path / "other.lfm")
    monkeypatch.setenv("LFM_B200_NO_PIPELINE", "1")                      # the references: the one-shot path
    L.write_stack(a, refa, nnum=13, **kwa)
    L.write_stack(b, refb, nnum=13, **kwb)
    monkeypatch.delenv("LFM_B200_NO_PIPELINE")
    c = lf_synth((12, 200, 230), 13, seed=13)
    L.write_stack(c, other, nnum=13, header_version=8 + 5, block_size=(64, 64, 4, 1, 1), way=0)
    blob = bytes(np.random.default_rng(3).integers(0, 4, 300000, dtype=np.uint8))
    import bz2
    wa = L.StackWriter(str(tmp_path / "a.lfm"), a.shape, nnum=13, **kwa)
    wb = L.StackWriter(str(tmp_path / "b.lfm"), b.shape, nnum=13, **kwb)
    db = _cuda(b)
    for i in range(45):
        wa.append(a[i])
        if i < 30:
            wb.append(db[i])
        if i % 7 == 3:
            assert np.array_equal(L.read_stack(other, way=0), c)
            assert torch.equal(L.read_stack(other, way=0, device="cuda").view(torch.int16), _cuda(c))
            assert L.bz2_compress(blob, 9) == bz2.compress(blob, 9)
    assert wb.close() == 30 and wa.close() == 45
    assert _md5(str(tmp_path / "a.lfm")) == _md5(refa)
    assert _md5(str(tmp_path / "b.lfm")) == _md5(refb)


# ---- bounded memory
def _rss():
    for line in open("/proc/self/status"):
        if line.startswith("VmRSS:"):
            return int(line.split()[1]) * 1024
    return 0


@pytest.mark.gpu
def test_memory_does_not_grow_with_the_recording(L, tmp_path):
    """512 frames of 2048^2 (4.3 GB) from a ring of 8 host frames: 12 frames per batch (>= 96 MB), so the device memory in use after
    16 batches may exceed its value after 2 batches by no more than 16 MB (allocator granularity), and the process RSS stays below
    the stack size"""
    import torch
    n, H, W = 512, 2048, 2048
    ring = lf_synth_int((8, H, W), 15, seed=3, device="cuda").cpu().numpy().view(np.uint16)
    d = "/dev/shm" if os.access("/dev/shm", os.W_OK) else str(tmp_path)
    fn = os.path.join(d, "lfm_rec_mem_%d.lfm" % os.getpid())
    per_batch = 12
    try:
        w = L.StackWriter(fn, (n, H, W), header_version=8 + 4, nnum=15, block_size=(96, 96, 1, 1, 1), way=2)
        free2 = free16 = None
        for f in range(n):
            w.append(ring[f % 8])
            if f == 2 * per_batch + 1:
                free2 = torch.cuda.mem_get_info()[0]
            if f == 16 * per_batch + 1:
                free16 = torch.cuda.mem_get_info()[0]
        assert _rss() < n * H * W * 2
        assert w.close() == n
        assert free2 - free16 <= 16 << 20, (free2, free16)
        assert np.array_equal(L.read_roi(fn, (0, 0, 509, 0, 0), (W - 1, H - 1, 511, 0, 0), way=2)[0, 0], ring[[5, 6, 7]])
    finally:
        if os.path.exists(fn):
            os.remove(fn)


# ---- no device
@pytest.mark.parametrize("fname", [None, b""])
def test_open_with_bad_arguments_is_code_3(Lhost, fname):
    w = C.c_void_p()
    rc = Lhost.lib.lfmStackWriterOpen(C.byref(w), fname, Lhost._xyzct((4, 60, 70)), 1, None, None, 1, None, 0, 13)
    assert rc == 3 and not w.value
    assert Lhost.lib.lfmStackWriterOpen(None, b"x.lfm", Lhost._xyzct((4, 60, 70)), 1, None, None, 1, None, 0, 13) == 3
    assert Lhost.lib.lfmStackWriterAppend(None, None, 1) == 3
    assert Lhost.lib.lfmStackWriterClose(None, None) == 3


@pytest.mark.skipif(has_cuda(), reason="checks the no-GPU behaviour")
def test_open_without_a_device_is_code_6_and_creates_no_file(Lhost, tmp_path):
    fn = str(tmp_path / "rec.lfm")
    with pytest.raises(Lhost.LfmError) as ei:
        Lhost.StackWriter(fn, (4, 60, 70))
    assert ei.value.code == 6
    assert not os.path.exists(fn)
