"""Device-resident .lfm files: write_stack from a CUDA tensor and read_stack / read_roi into GPU memory (writeLFMstackDevice,
readLFMroiDevice in include/lfm_b200.h).  The file written from the device must be byte-identical to the one written from the
numpy copy of the same stack, and the pixels decoded into GPU memory must equal what the host reads return."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, has_cuda, lf_synth, lf_synth_int


@pytest.fixture(scope="module")
def L():
    import lfm_b200
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    lfm_b200.set_devices(0, 1)
    return lfm_b200


def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda()


def _host(t):
    """a CUDA uint16 / int16 tensor -> numpy uint16 (compared through the int16 view: torch has few uint16 operations)"""
    import torch
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def _pair_runs(shape, seed):
    """lf_synth with a corner of pixel pairs (4-byte runs): cut into 160x160x8 blocks, some streams hold two bzip2 blocks"""
    rng = np.random.default_rng(12)
    a = lf_synth(shape, 13, seed=seed)
    a[:, :150, :170] = np.repeat(rng.integers(0, 60000, (shape[0], 150, 85)), 2, axis=2).astype(np.uint16)
    return a


# name: (stack, write_stack keyword arguments, LFM_B200_BATCH_KB or None)
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
    c["channels_times_blocked"] = (lambda: lf_synth((30, 60, 70), 13, seed=3).reshape(2, 3, 5, 60, 70),
                                   dict(header_version=8 + 4, block_size=(32, 32, 2, 2, 1), way=0), None)
    c["codec_none"] = (lambda: lf_synth((7, 150, 170), 13, seed=9), dict(header_version=8 + 5, block_size=(64, 48, 4, 1, 1), way=0, codec=0), None)
    c["slab_pipeline_auto"] = (lambda: lf_synth((45, 200, 230), 13, seed=11), dict(header_version=0, block_size=(64, 64, 4, 1, 1), way=0), 400)
    c["slab_pipeline_video"] = (lambda: lf_synth((45, 200, 230), 13, seed=11), dict(header_version=0x80 | 12, block_size=(64, 64, 3, 1, 1), way=0), 300)
    c["slab_pipeline_raw"] = (lambda: lf_synth((45, 200, 230), 13, seed=11), dict(header_version=8, block_size=(96, 96, 1, 1, 1), way=0), 100)
    return c


CASES = _cases()


def _boxes(shape5):
    """ROIs (lb, ub) in x,y,z,c,t: XZ and YZ planes, a box from an odd frame, single pixels, and boxes across c and t"""
    t, c, z, y, x = shape5
    full_ct = ((0, 0), (c - 1, t - 1))
    b = []
    for (c0, t0), (c1, t1) in (full_ct, ((c - 1, t - 1), (c - 1, t - 1))):
        b += [((0, y // 2, 0, c0, t0), (x - 1, y // 2, z - 1, c1, t1)),                     # XZ plane
              ((x // 3, 0, 0, c0, t0), (x // 3, y - 1, z - 1, c1, t1)),                     # YZ plane
              ((3, 5, min(1, z - 1), c0, t0), (x - 2, y - 7, z - 1, c1, t1)),              # from an odd frame
              ((x - 1, y - 1, z - 1, c0, t0), (x - 1, y - 1, z - 1, c0, t0))]
    b.append(((0, 0, 0, 0, 0), (x - 1, y - 1, z - 1, c - 1, t - 1)))                       # the whole stack as a box
    return b


def _shape5(a):
    s = list(a.shape)
    while len(s) < 5:
        s.insert(0, 1)
    return tuple(s)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_device_write_is_byte_identical_and_device_reads_match(L, tmp_path, monkeypatch, name):
    import torch
    make, kw, batch_kb = CASES[name]
    if batch_kb:
        monkeypatch.setenv("LFM_B200_BATCH_KB", str(batch_kb))          # slab pipeline on both sides
    a = make()
    fh, fd = str(tmp_path / "host.lfm"), str(tmp_path / "dev.lfm")
    L.write_stack(a, fh, nnum=13, **kw)
    t = _cuda(a)
    L.write_stack(t, fd, nnum=13, **kw)
    assert L.stats().ms_h2d == 0
    assert open(fd, "rb").read() == open(fh, "rb").read(), name
    way = kw["way"]
    host = L.read_stack(fh, way=way)
    dev = L.read_stack(fd, way=way, device="cuda")
    assert L.stats().ms_d2h == 0
    assert dev.dtype == torch.uint16 and dev.is_cuda and tuple(dev.shape) == host.shape
    assert torch.equal(dev.view(torch.int16), t.view(dev.shape)), name
    out = torch.full(host.shape, 7, dtype=torch.int16, device="cuda")
    assert L.read_stack(fd, way=way, out=out) is out
    assert np.array_equal(_host(out), host)
    for lb, ub in _boxes(_shape5(a)):
        want = L.read_roi(fh, lb, ub, way=way)
        got = L.read_roi(fd, lb, ub, way=way, device="cuda")
        assert L.stats().ms_d2h == 0
        assert tuple(got.shape) == want.shape and np.array_equal(_host(got), want), (name, lb, ub)


@pytest.mark.gpu
def test_device_write_pixel_size_and_metadata(L, tmp_path):
    a = lf_synth((6, 90, 110), 13, seed=2)
    t = _cuda(a)
    ps = (C.c_float * 5)(0.5, 0.25, 2.0, 1.0, 3.0)
    meta = C.create_string_buffer(b"device-resident write, pixel size 0.5 x 0.25 x 2", 256)
    bs = L._u32x5(64, 32, 2, 1, 1)
    fh, fd = os.fsencode(str(tmp_path / "h.lfm")), os.fsencode(str(tmp_path / "d.lfm"))
    args = (L._xyzct(a.shape), 1, -1, C.cast(ps, C.c_void_p), C.cast(bs, C.c_void_p), 1, C.cast(meta, C.c_void_p), 8 + 6, 13)
    L.set_way(0)
    assert L.lib.writeLFMstackEx(a.ctypes.data, fh, *args) == 0
    assert L.lib.writeLFMstackDevice(t.data_ptr(), fd, *args) == 0
    assert open(fd, "rb").read() == open(fh, "rb").read()
    h = L.read_header(fd)
    assert h["pixelSize"] == [0.5, 0.25, 2.0, 1.0, 3.0] and h["metadata"] == meta.raw
    assert np.array_equal(_host(L.read_stack(fd, way=0, device="cuda")), a)


@pytest.mark.gpu
def test_device_write_on_two_gpus_setting(L, tmp_path):
    """lfmSetDevices(0, 2): the device calls run on the first device alone; the file equals the one-GPU file"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    a = lf_synth((24, 100, 120), 13, seed=2)
    fh, fd = str(tmp_path / "h.lfm"), str(tmp_path / "d.lfm")
    L.write_stack(a, fh, header_version=0x80 | 13, nnum=13, block_size=(48, 48, 4, 1, 1), way=0)
    t = _cuda(a)
    try:
        assert L.set_devices(0, 2) == 2
        L.write_stack(t, fd, header_version=0x80 | 13, nnum=13, block_size=(48, 48, 4, 1, 1), way=0)
        assert open(fd, "rb").read() == open(fh, "rb").read()
        assert torch.equal(L.read_stack(fd, way=0, device="cuda").view(torch.int16), t)
        r = L.read_roi(fd, (5, 6, 3, 0, 0), (90, 70, 20, 0, 0), way=0, device="cuda")
        assert np.array_equal(_host(r)[0, 0], a[3:21, 6:71, 5:91])
    finally:
        L.set_devices(0, 1)


@pytest.mark.gpu
def test_device_reads_of_oracle_files(L, oracle, tmp_path):
    """files the CPU oracle writes decode into GPU memory as the host reads decode them"""
    a = lf_synth((12, 110, 140), 13, seed=21)
    fn = str(tmp_path / "o.lfm")
    for hv, way, bs in ((0, 0, (64, 64, 4, 1, 1)), (8 + 3, 1, (48, 64, 5, 1, 1)), (0x80 | 13, 0, (64, 64, 3, 1, 1)), (8, 2, None)):
        rc, _ = oracle.write(a, fn, hv, 13, way, block_size=bs)
        assert rc == 0
        assert np.array_equal(_host(L.read_stack(fn, way=way, device="cuda")), a), (hv, way)
        for lb, ub in _boxes(_shape5(a)):
            assert np.array_equal(_host(L.read_roi(fn, lb, ub, way=way, device="cuda")), L.read_roi(fn, lb, ub, way=way)), (hv, way, lb, ub)


@pytest.mark.gpu
def test_device_rois_of_the_host_roi_tests(L, tmp_path):
    """the boxes of test_roi_without_predictor_decodes_only_needed_blocks (predictor off, then video) and the c5-slice boxes"""
    a = lf_synth((20, 120, 130), 13, seed=8)
    fn = str(tmp_path / "r.lfm")
    L.write_stack(_cuda(a), fn, header_version=8, block_size=(32, 32, 4, 1, 1), way=0)
    for lb, ub in [((0, 0, 7, 0, 0), (129, 119, 7, 0, 0)), ((40, 0, 0, 0, 0), (40, 119, 19, 0, 0)), ((3, 50, 2, 0, 0), (77, 50, 17, 0, 0)),
                   ((33, 31, 3, 0, 0), (64, 95, 12, 0, 0))]:
        r = L.read_roi(fn, lb, ub, device="cuda")
        assert np.array_equal(_host(r)[0, 0], a[lb[2]:ub[2] + 1, lb[1]:ub[1] + 1, lb[0]:ub[0] + 1])
    L.write_stack(_cuda(a), fn, header_version=0x80 | 12, block_size=(32, 32, 4, 1, 1), way=0)
    r = L.read_roi(fn, (10, 20, 5, 0, 0), (100, 90, 9, 0, 0), device="cuda")
    assert np.array_equal(_host(r)[0, 0], a[5:10, 20:91, 10:101])
    # c5 slice: 16 x 4096 x 4096, tiles, auto-select
    t = lf_synth_int((16, 4096, 4096), 13, seed=7, device="cuda")
    fn = str(tmp_path / "c5s.lfm")
    L.write_stack(t, fn, header_version=0, nnum=13, way=0)
    for lb, ub in (((0, 0, 5), (4095, 4095, 5)), ((1700, 1800, 3), (2211, 2311, 12))):
        r = L.read_roi(fn, lb + (0, 0), ub + (0, 0), way=0, device="cuda")
        assert np.array_equal(_host(r)[0, 0], _host(t[lb[2]:ub[2] + 1, lb[1]:ub[1] + 1, lb[0]:ub[0] + 1]))
        assert np.array_equal(_host(r), L.read_roi(fn, lb + (0, 0), ub + (0, 0), way=0))


def _fullsize_golden():
    fn = os.path.join(GOLDEN, "fullsize.json")
    return json.load(open(fn)) if os.path.exists(fn) else {}


def _scratch_file(tmp_path, name, nbytes):
    """/dev/shm when it has room for the file (tmpfs: the file write is a memory copy), else the test's directory"""
    if os.path.isdir("/dev/shm"):
        st = os.statvfs("/dev/shm")
        if st.f_bavail * st.f_frsize > 2 * nbytes:
            return os.path.join("/dev/shm", "lfm_devio_%d_%s" % (os.getpid(), name))
    return str(tmp_path / name)


FULL = {"c3": ((101, 2048, 2048), 13, 1, 0), "c4": ((1000, 1024, 1024), 13, 0, 0x80), "c5": ((200, 4096, 4096), 13, 0, 0)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FULL))
def test_full_size_device_write_md5_and_device_read(L, tmp_path, name):
    """BASELINE full-size configs generated on the GPU and written from there: the file has the md5 the reference's file has
    (tests/golden/fullsize.json), and reading it back into GPU memory gives the input tensor.  No pixel crosses PCIe."""
    import torch
    G = _fullsize_golden()
    if name not in G:
        pytest.skip("no committed md5 for %s (tests/golden/fullsize.json)" % name)
    shape, nnum, way, hv = FULL[name]
    g = G[name]
    t = lf_synth_int(shape, nnum, seed=7, device="cuda")
    hv_req = hv if g["stored_hv"] == g.get("engine_stored_hv", g["stored_hv"]) else (hv & 0x80) | (8 + (g["stored_hv"] & 0x7F))
    fn = _scratch_file(tmp_path, name + ".lfm", g["size"])
    try:
        L.write_stack(t, fn, header_version=hv_req, nnum=nnum, way=way)
        assert L.stats().ms_h2d == 0
        assert os.path.getsize(fn) == g["size"]
        md5 = hashlib.md5()
        with open(fn, "rb") as f:
            for chunk in iter(lambda: f.read(64 << 20), b""):
                md5.update(chunk)
        assert md5.hexdigest() == g["md5"], "%s: file differs from the reference's" % name
        back = L.read_stack(fn, way=way, device="cuda")
        assert L.stats().ms_d2h == 0
        assert torch.equal(back.view(torch.int16), t)
    finally:
        if os.path.exists(fn):
            os.remove(fn)


@pytest.mark.gpu
def test_device_io_errors(L, tmp_path):
    import torch
    a = lf_synth((6, 70, 90), 13, seed=5)
    t = _cuda(a)
    fn = str(tmp_path / "e.lfm")
    L.write_stack(t, fn, header_version=8 + 2, block_size=(32, 32, 2, 1, 1), way=0)
    fb = os.fsencode(fn)
    n = C.c_uint64()
    # capacity: one byte short -> 5, size reported, nothing written (guard bytes around the buffer too); exact -> the pixels
    lb, ub = L._u32x5(4, 3, 1, 0, 0), L._u32x5(80, 60, 4, 0, 0)
    box = a[1:5, 3:61, 4:81]
    G = 4096
    buf = torch.full((box.nbytes + 2 * G,), 0x5A, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr() + G
    assert L.lib.readLFMroiDevice(fb, lb, ub, p, box.nbytes - 1, C.byref(n)) == 5
    assert n.value == box.nbytes
    assert bool((buf == 0x5A).all())
    assert L.lib.readLFMroiDevice(fb, lb, ub, p, box.nbytes, C.byref(n)) == 0 and n.value == box.nbytes
    assert bool((buf[:G] == 0x5A).all()) and bool((buf[G + box.nbytes:] == 0x5A).all())
    assert np.array_equal(buf[G:G + box.nbytes].cpu().numpy().view(np.uint16).reshape(box.shape), box)
    # whole-file reads below go to a buffer of the whole stack's size: a code other than 5 is not a capacity refusal
    whole = torch.full((a.nbytes,), 0x5A, dtype=torch.uint8, device="cuda")
    assert L.lib.readLFMroiDevice(fb, None, None, whole.data_ptr(), a.nbytes - 1, C.byref(n)) == 5 and n.value == a.nbytes
    assert bool((whole == 0x5A).all())
    # host memory is not a device buffer
    h = np.empty_like(a)
    assert L.lib.readLFMroiDevice(fb, None, None, h.ctypes.data, h.nbytes, C.byref(n)) == 3
    xyzct = L._xyzct(a.shape)
    assert L.lib.writeLFMstackDevice(a.ctypes.data, os.fsencode(str(tmp_path / "h.lfm")), xyzct, 1, -1, None, None, 1, None, 8, 13) == 3
    # a tensor on another GPU
    if torch.cuda.device_count() >= 2:
        t1 = t.to("cuda:1")
        with pytest.raises(L.LfmError) as ei:
            L.write_stack(t1, str(tmp_path / "g1.lfm"), header_version=8, way=0)
        assert ei.value.code == 3
        with pytest.raises(L.LfmError) as ei:
            L.read_stack(fn, way=0, out=torch.empty_like(t1))
        assert ei.value.code == 3
    # ZLIB and 8-bit pixels: 7, writing and reading
    assert L.lib.writeLFMstackDevice(t.data_ptr(), os.fsencode(str(tmp_path / "z.lfm")), xyzct, 1, -1, None, None, 2, None, 8, 13) == 7
    assert L.lib.writeLFMstackDevice(t.data_ptr(), os.fsencode(str(tmp_path / "u8.lfm")), xyzct, 0, -1, None, None, 1, None, 8, 13) == 7
    good = open(fn, "rb").read()
    for off, val in ((43, 2), (42, 0)):
        raw = bytearray(good); raw[off] = val
        bad = str(tmp_path / "b.lfm"); open(bad, "wb").write(bytes(raw))
        assert L.lib.readLFMroiDevice(os.fsencode(bad), None, None, whole.data_ptr(), whole.numel(), C.byref(n)) == 7, (off, val)
    # truncated file, flipped payload byte: 2
    bad = str(tmp_path / "b.lfm")
    open(bad, "wb").write(good[:-100])
    assert L.lib.readLFMroiDevice(os.fsencode(bad), None, None, whole.data_ptr(), whole.numel(), C.byref(n)) == 2
    raw = bytearray(good); raw[len(raw) - 200] ^= 0x5A
    open(bad, "wb").write(bytes(raw))
    with pytest.raises(L.LfmError) as ei:
        L.read_stack(bad, way=0, device="cuda")
    assert ei.value.code == 2
    # box outside the stack: 3; missing file: 3; file that cannot be created: 5
    assert L.lib.readLFMroiDevice(fb, L._u32x5(0, 0, 0, 0, 0), L._u32x5(90, 69, 5, 0, 0), whole.data_ptr(), whole.numel(), C.byref(n)) == 3
    with pytest.raises(L.LfmError) as ei:
        L.read_roi(fn, (0, 0, 5, 0, 0), (10, 10, 6, 0, 0), way=0, device="cuda")
    assert ei.value.code == 3
    assert L.lib.readLFMroiDevice(os.fsencode(str(tmp_path / "missing.lfm")), None, None, whole.data_ptr(), whole.numel(), C.byref(n)) == 3
    with pytest.raises(L.LfmError) as ei:
        L.write_stack(t, "/nonexistent_dir/x.lfm", header_version=8)
    assert ei.value.code == 5
    # a wrong-sized out= tensor is refused before the call
    with pytest.raises(ValueError):
        L.read_stack(fn, way=0, out=torch.empty(7, dtype=torch.int16, device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("way,hv,batch_kb", [(2, 8 + 4, None), (2, 8 + 1, None), (2, 8 + 2, None), (2, 8 + 4, 100), (1, 8 + 3, None),
                                             (0, 0x80 | 12, None), (0, 8, None), (0, 8, 100)])
def test_device_reads_into_buffers_at_any_offset(L, tmp_path, monkeypatch, way, hv, batch_kb):
    """out= views into a workspace start at any even byte offset, not only at the 16-byte alignment of torch's allocations: frames
    2048 / 1024 bytes wide make the decode and inverse-predictor kernels take their 16-byte vector paths (way space predictors 1, 2, 4:
    the prefix-sum kernels), the slab pipeline included.  Every offset gets the exact pixels, the workspace around them is untouched."""
    import torch
    if batch_kb:
        monkeypatch.setenv("LFM_B200_BATCH_KB", str(batch_kb))
    shape = (9, 256, 512) if not (hv & 0x80) else (9, 128, 1024)
    a = lf_synth(shape, 15, seed=6)
    bs = (64, 64, 3 if hv & 0x80 else 2, 1, 1)
    fn = str(tmp_path / "o.lfm")
    L.write_stack(a, fn, header_version=hv, nnum=15, block_size=bs, way=way)
    n = a.size
    ws = torch.full((n + 64,), -21555, dtype=torch.int16, device="cuda")
    for off in (0, 1, 2, 3, 4, 7, 8):
        ws.fill_(-21555)
        out = ws[off:off + n].view(shape)
        assert L.read_stack(fn, way=way, out=out) is out
        assert np.array_equal(_host(out), a), (way, hex(hv), off)
        assert bool((ws[:off] == -21555).all()) and bool((ws[off + n:] == -21555).all()), (way, hex(hv), off)
        lb, ub = (3, 5, 1, 0, 0), (shape[2] - 9, shape[1] - 2, 7, 0, 0)
        box = a[1:8, 5:shape[1] - 1, 3:shape[2] - 8]
        r = ws[off:off + box.size].view((1, 1) + box.shape)
        assert L.read_roi(fn, lb, ub, way=way, out=r) is r
        assert np.array_equal(_host(r)[0, 0], box), (way, hex(hv), off)


@pytest.mark.gpu
def test_device_and_out_must_agree(L, tmp_path):
    import torch
    a = lf_synth((2, 40, 48), 13, seed=1)
    fn = str(tmp_path / "d.lfm")
    L.write_stack(a, fn, header_version=8, way=0)
    out = torch.empty(a.shape, dtype=torch.int16, device="cuda")
    assert L.read_stack(fn, way=0, device="cuda", out=out) is out and np.array_equal(_host(out), a)
    with pytest.raises(ValueError):
        L.read_stack(fn, way=0, device="cpu", out=out)
    if torch.cuda.device_count() >= 2:
        with pytest.raises(ValueError):
            L.read_stack(fn, way=0, device="cuda:1", out=out)


@pytest.mark.skipif(has_cuda(), reason="checks the no-GPU behaviour")
def test_device_file_calls_without_gpu(oracle, tmp_path):
    """without a CUDA device the device-resident file calls fail with code 6, as the host calls do"""
    import lfm_b200 as M
    a = lf_synth((2, 40, 40), 13)
    fn = str(tmp_path / "o.lfm")
    rc, _ = oracle.write(a, fn, 8, 13, 0)
    assert rc == 0
    xyzct = M._u32x5(40, 40, 2, 1, 1)
    assert M.lib.writeLFMstackDevice(a.ctypes.data, os.fsencode(str(tmp_path / "x.lfm")), xyzct, 1, -1, None, None, 1, None, 8, 13) == 6
    assert M.lib.writeLFMstackDevice(a.ctypes.data, b"/nonexistent_dir/x.lfm", xyzct, 1, -1, None, None, 1, None, 8, 13) == 5
    n = C.c_uint64()
    assert M.lib.readLFMroiDevice(os.fsencode(fn), None, None, a.ctypes.data, a.nbytes, C.byref(n)) == 6
    assert M.lib.readLFMroiDevice(os.fsencode(fn), M._u32x5(0, 0, 0, 0, 0), M._u32x5(9, 9, 1, 0, 0), a.ctypes.data, a.nbytes, C.byref(n)) == 6
    assert M.lib.readLFMroiDevice(os.fsencode(str(tmp_path / "missing.lfm")), None, None, a.ctypes.data, a.nbytes, C.byref(n)) == 3
