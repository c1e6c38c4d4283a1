"""Playing a stack back frame by frame (StackReader; lfmStackReaderOpen / Read / ReadDevice / Close in include/lfm_b200.h).
Whatever the box, the read chunking and the destination (numpy, CUDA tensors, out= views at odd offsets, host and device reads
mixed), the frames a reader hands out must be the pixels read_stack / read_roi return for the same box of the same file."""
import ctypes as C
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from conftest import has_cuda, lf_synth
from test_stack_writer import CASES, _frames

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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


def _host(t):
    import torch
    return t.view(torch.int16).cpu().numpy().view(np.uint16)


def _shape5(a):
    return a.shape if a.ndim == 5 else (1, 1) + a.shape


def _boxes(shape5):
    """(name, lb, ub): the whole stack, a range starting at an odd frame, an x/y crop, a z sub-range, a single frame"""
    T, Cn, Z, Y, X = shape5
    full_ub = (X - 1, Y - 1, Z - 1, Cn - 1, T - 1)
    out = [("whole", None, None)]
    if T > 1:
        out.append(("t_from_1", (0, 0, 0, 0, 1), full_ub))                # frame Z * C: odd for odd volumes
    else:
        out.append(("z_from_odd", (0, 0, 3, 0, 0), full_ub))
    out.append(("xy_crop", (5, 3, 0, 0, 0), (X - 9, Y - 4, Z - 1, Cn - 1, T - 1)))
    if Z > 2:
        out.append(("z_sub", (7, 0, 1, 0, 0), (X - 1, Y - 6, min(Z - 1, 3), Cn - 1, T - 1)))
    out.append(("one_frame", (0, 0, Z // 2, Cn - 1, T - 1), (X - 1, Y - 1, Z // 2, Cn - 1, T - 1)))
    return out


def _crop(a5, lb, ub):
    if lb is None:
        return a5
    return a5[lb[4]:ub[4] + 1, lb[3]:ub[3] + 1, lb[2]:ub[2] + 1, lb[1]:ub[1] + 1, lb[0]:ub[0] + 1]


def _play(L, fn, lb, ub, way, chunk, sink):
    """every frame of the box through one reader: reads of `chunk` frames (0: all at once) into `sink`"""
    import torch
    out = []
    with L.StackReader(fn, lb, ub, way=way, device="cuda" if sink == "cuda" else None) as r:
        F, Y, X = r.shape
        n = chunk or F
        i = 0
        while True:
            if sink == "view" or (sink == "alternate" and i % 2 == 1):
                ws = torch.full((n * Y * X + 9,), -21555, dtype=torch.int16, device="cuda")
                part = r.read(n, out=ws[1:1 + n * Y * X].view(n, Y, X))         # 2 bytes into the allocation
                assert bool((ws[0] == -21555).all()) and bool((ws[1 + n * Y * X:] == -21555).all())
                part = _host(part)
            elif sink == "cuda":
                part = _host(r.read(n))
            else:
                part = r.read(n)
            i += 1
            if len(part) == 0:
                break
            assert len(part) == n or sum(len(p) for p in out) + len(part) == F
            out.append(part)
        assert len(r.read(3)) == 0                                        # past the end: nothing, and the reader stays usable
    return np.concatenate(out) if out else np.zeros((0,), np.uint16)


def _check_file(L, fn, a, way):
    a5 = a.reshape(_shape5(a))
    assert np.array_equal(L.read_stack(fn, way=way).reshape(a5.shape), a5)
    for name, lb, ub in _boxes(a5.shape):
        want = _crop(a5, lb, ub)
        if lb is not None:
            try:
                assert np.array_equal(L.read_roi(fn, lb, ub, way=way), want), name
            except L.LfmError as e:
                # an ROI read refuses a box whose first slab starts on an odd frame after another such slab (the middle of an
                # odd video volume): the reader decodes those slabs, and its frames are checked against read_stack alone
                assert e.code == 7 and a5.shape[2] % 2 == 1, name
        want = want.reshape(-1, want.shape[-2], want.shape[-1])
        for chunk in (1, 7, 0):
            for sink in ("numpy", "cuda", "view", "alternate"):
                got = _play(L, fn, lb, ub, way, chunk, sink)
                assert got.shape == want.shape and np.array_equal(got, want), (name, chunk, sink)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_playback_matches_read_roi(L, tmp_path, monkeypatch, name):
    make, kw, batch_kb = CASES[name]
    if batch_kb:
        monkeypatch.setenv("LFM_B200_BATCH_KB", str(batch_kb))          # batches of a few slabs
    a = make()
    fn = str(tmp_path / "s.lfm")
    L.write_stack(a, fn, nnum=13, **kw)
    _check_file(L, fn, a, kw["way"])


@pytest.mark.gpu
def test_playback_of_oracle_files_and_early_closed_recordings(L, oracle, tmp_path, monkeypatch):
    a = lf_synth((12, 110, 140), 13, seed=21)
    fn = str(tmp_path / "o.lfm")
    for hv, way, bs in ((0, 0, (64, 64, 4, 1, 1)), (8 + 3, 1, (48, 64, 5, 1, 1)), (0x80 | 13, 0, (64, 64, 3, 1, 1))):
        rc, _ = oracle.write(a, fn, hv, 13, way, block_size=bs)
        assert rc == 0
        _check_file(L, fn, a, way)
    monkeypatch.setenv("LFM_B200_BATCH_KB", "60")
    v = lf_synth((40, 100, 120), 13, seed=14).reshape(8, 1, 5, 100, 120)
    rec = str(tmp_path / "rec.lfm")
    w = L.StackWriter(rec, v.shape, header_version=0x80 | 12, nnum=13, block_size=(64, 64, 2, 1, 1), way=0)
    w.append(_frames(v)[:23])
    assert w.close() == 20
    _check_file(L, rec, v[:4], 0)


@pytest.mark.gpu
def test_host_reads_stay_inside_dst(L, tmp_path, monkeypatch):
    monkeypatch.setenv("LFM_B200_BATCH_KB", "100")
    a = lf_synth((20, 120, 130), 13, seed=8)
    fn = str(tmp_path / "g.lfm")
    L.write_stack(a, fn, header_version=8 + 4, block_size=(32, 32, 2, 1, 1), way=0)
    lb, ub = L._u32x5(3, 5, 2, 0, 0), L._u32x5(100, 90, 17, 0, 0)
    box = a[2:18, 5:91, 3:101]
    r = C.c_void_p(); frames = C.c_uint64(); fb = C.c_uint64(); got = C.c_uint64()
    assert L.lib.lfmStackReaderOpen(C.byref(r), os.fsencode(fn), lb, ub, C.byref(frames), C.byref(fb)) == 0
    assert frames.value == 16 and fb.value == box[0].nbytes
    G = 4096
    buf = np.full(box.nbytes + 2 * G, 0x5A, np.uint8)
    pos = 0
    for n in (5, 1, 7, 9):
        assert L.lib.lfmStackReaderRead(r, buf.ctypes.data + G + pos, n, C.byref(got)) == 0
        assert got.value == min(n, 16 - pos // fb.value)
        pos += got.value * fb.value
    assert L.lib.lfmStackReaderRead(r, buf.ctypes.data, 4, C.byref(got)) == 0 and got.value == 0
    assert (buf[:G] == 0x5A).all() and (buf[G + box.nbytes:] == 0x5A).all()
    assert np.array_equal(buf[G:G + box.nbytes].view(np.uint16).reshape(box.shape), box)
    assert L.lib.lfmStackReaderClose(r) == 0


# ---- errors
def _open(L, fn, lb=None, ub=None):
    r = C.c_void_p(); frames = C.c_uint64(); fb = C.c_uint64()
    rc = L.lib.lfmStackReaderOpen(C.byref(r), fn, lb, ub, C.byref(frames), C.byref(fb))
    return rc, r


def _reader_code(L, fn, lb=None, ub=None, nbytes=1 << 22):
    """Open's code, or the code of reading every frame into device memory, or 0"""
    import torch
    rc, r = _open(L, fn, lb, ub)
    if rc:
        assert not r.value
        return rc
    buf = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    got = C.c_uint64()
    rc = L.lib.lfmStackReaderReadDevice(r, buf.data_ptr(), 1 << 20, C.byref(got))
    rc2 = L.lib.lfmStackReaderClose(r)
    assert rc2 == rc
    return rc


@pytest.mark.gpu
def test_error_codes_match_read_lfm_roi_device(L, tmp_path):
    import torch
    a = lf_synth((6, 70, 90), 13, seed=5)
    fn = str(tmp_path / "e.lfm")
    L.write_stack(a, fn, header_version=8 + 2, block_size=(32, 32, 2, 1, 1), way=0)
    whole = torch.empty(a.nbytes, dtype=torch.uint8, device="cuda")
    n = C.c_uint64()

    def roi_code(f, lb=None, ub=None):
        return L.lib.readLFMroiDevice(os.fsencode(f), lb, ub, whole.data_ptr(), whole.numel(), C.byref(n))

    good = open(fn, "rb").read()
    files = []
    for off, val in ((43, 2), (42, 0)):                                   # ZLIB, 8-bit pixels: 7
        raw = bytearray(good); raw[off] = val
        files.append(("hdr%d" % off, bytes(raw)))
    files.append(("truncated", good[:-100]))
    raw = bytearray(good); raw[len(raw) - 200] ^= 0x5A
    files.append(("flipped", bytes(raw)))
    for what, data in files:
        bad = str(tmp_path / (what + ".lfm")); open(bad, "wb").write(data)
        want = roi_code(bad)
        assert want in (2, 7), what
        assert _reader_code(L, os.fsencode(bad)) == want, what
    boxes = [(L._u32x5(0, 0, 0, 0, 0), L._u32x5(90, 69, 5, 0, 0)), (L._u32x5(0, 0, 5, 0, 0), L._u32x5(10, 10, 6, 0, 0)),
             (L._u32x5(5, 0, 0, 0, 0), L._u32x5(4, 10, 1, 0, 0))]
    for lb, ub in boxes:
        assert roi_code(fn, lb, ub) == 3
        assert _reader_code(L, os.fsencode(fn), lb, ub) == 3
    missing = str(tmp_path / "missing.lfm")
    assert roi_code(missing) == 3 and _reader_code(L, os.fsencode(missing)) == 3
    assert _open(L, b"")[0] == 3 and _open(L, None)[0] == 3
    assert _open(L, os.fsencode(fn), L._u32x5(0, 0, 0, 0, 0), None)[0] == 3
    # video written with way 1 and read with way 0 / way 1
    v = str(tmp_path / "v.lfm")
    L.write_stack(a, v, header_version=0x80 | 12, block_size=(32, 32, 2, 1, 1), way=0)
    L.set_way(1)
    try:
        assert roi_code(v) == 7 and _reader_code(L, os.fsencode(v)) == 7
    finally:
        L.set_way(0)
    # c/t-blocked files: readable as a whole, but not as a stream
    b = lf_synth((30, 60, 70), 13, seed=3).reshape(2, 3, 5, 60, 70)
    for bs in ((32, 32, 2, 2, 1), (32, 32, 2, 1, 2)):
        L.write_stack(b, fn, header_version=8 + 4, block_size=bs, way=0)
        assert np.array_equal(L.read_stack(fn, way=0), b)
        with pytest.raises(L.LfmError) as ei:
            L.StackReader(fn, way=0)
        assert ei.value.code == 7
    # a bad destination fails the reader with 3
    L.write_stack(a, fn, header_version=8 + 2, block_size=(32, 32, 2, 1, 1), way=0)
    rc, r = _open(L, os.fsencode(fn))
    assert rc == 0
    h = np.empty(a.shape, np.uint16)
    got = C.c_uint64()
    assert L.lib.lfmStackReaderReadDevice(r, h.ctypes.data, 1, C.byref(got)) == 3 and got.value == 0
    assert L.lib.lfmStackReaderRead(r, h.ctypes.data, 1, C.byref(got)) == 3
    assert L.lib.lfmStackReaderClose(r) == 3
    rc, r = _open(L, os.fsencode(fn))
    assert L.lib.lfmStackReaderRead(r, None, 1, C.byref(got)) == 3
    assert L.lib.lfmStackReaderClose(r) == 3


@pytest.mark.gpu
def test_file_truncated_after_open_fails_with_2(L, tmp_path, monkeypatch):
    monkeypatch.setenv("LFM_B200_BATCH_KB", "100")
    a = lf_synth((40, 120, 130), 13, seed=2)
    fn = str(tmp_path / "t.lfm")
    L.write_stack(a, fn, header_version=8 + 4, block_size=(32, 32, 1, 1, 1), way=0)
    table = 320 + 8 * L.lib.lfmNumBlocks(L._xyzct(a.shape), C.cast(L._bs((32, 32, 1, 1, 1)), C.c_void_p))
    rc, r = _open(L, os.fsencode(fn))
    assert rc == 0
    os.truncate(fn, table + 1000)
    G = 4096
    buf = np.full(a.nbytes + 2 * G, 0x5A, np.uint8)
    got = C.c_uint64()
    assert L.lib.lfmStackReaderRead(r, buf.ctypes.data + G, 40, C.byref(got)) == 2 and got.value == 0
    assert (buf[:G] == 0x5A).all() and (buf[G + a.nbytes:] == 0x5A).all()
    assert L.lib.lfmStackReaderRead(r, buf.ctypes.data + G, 1, C.byref(got)) == 2
    assert L.lib.lfmStackReaderClose(r) == 2


# ---- sharing
@pytest.mark.gpu
def test_two_readers_a_writer_and_other_calls_between_reads(L, tmp_path, monkeypatch):
    import bz2
    import torch
    monkeypatch.setenv("LFM_B200_BATCH_KB", "300")
    a = lf_synth((45, 200, 230), 13, seed=11)
    b = lf_synth((30, 150, 170), 13, seed=12)
    fa, fb, fw = str(tmp_path / "a.lfm"), str(tmp_path / "b.lfm"), str(tmp_path / "w.lfm")
    L.write_stack(a, fa, nnum=13, header_version=0, block_size=(64, 64, 4, 1, 1), way=0)
    L.write_stack(b, fb, nnum=13, header_version=0x80 | 12, block_size=(64, 64, 3, 1, 1), way=0)
    blob = bytes(np.random.default_rng(3).integers(0, 4, 300000, dtype=np.uint8))
    ra = L.StackReader(fa, way=0)
    rb = L.StackReader(fb, (3, 4, 1, 0, 0), (160, 140, 29, 0, 0), way=0, device="cuda")
    w = L.StackWriter(fw, b.shape, nnum=13, header_version=8 + 4, block_size=(64, 64, 3, 1, 1), way=0)
    got_a, got_b = [], []
    for i in range(45):
        got_a.append(ra.read(1))
        if i < 30:
            got_b.append(_host(rb.read(1)))
            w.append(b[i])
        if i % 7 == 3:
            assert L.bz2_compress(blob, 9) == bz2.compress(blob, 9)
            assert np.array_equal(L.read_stack(fb, way=0), b)
            assert torch.equal(L.read_stack(fa, way=0, device="cuda").view(torch.int16), torch.from_numpy(a.view(np.int16)).cuda())
    assert len(ra.read(1)) == 0 and len(rb.read(1)) == 0
    ra.close(); rb.close()
    assert w.close() == 30
    assert np.array_equal(np.concatenate(got_a), a)
    assert np.array_equal(np.concatenate(got_b), b[1:, 4:141, 3:161])
    assert np.array_equal(L.read_stack(fw, way=0), b)


# ---- bounded memory
_MEM_CHILD = textwrap.dedent("""
    import os, sys, json
    import numpy as np
    import torch
    sys.path.insert(0, sys.argv[1])
    import lfm_b200 as L
    L.set_devices(0, 1)
    n, H, W = 4000, 64, 96
    fn = sys.argv[2]
    ring = (np.arange(16 * H * W, dtype=np.uint32) * 2654435761 % 997).astype(np.uint16).reshape(16, H, W)
    with L.StackWriter(fn, (n, H, W), header_version=8 + 4, nnum=13, block_size=(32, 32, 1, 1, 1), way=0) as w:
        for f in range(n):
            w.append(ring[f % 16])
    def rss():
        for line in open("/proc/self/status"):
            if line.startswith("VmRSS:"):
                return int(line.split()[1]) * 1024
    marks = {}
    with L.StackReader(fn, way=0) as r:
        for f in range(n):
            fr = r.read(1) if f % 2 == 0 else r.read(1, out=torch.empty((1, H, W), dtype=torch.uint16, device="cuda")).cpu().numpy()
            assert np.array_equal(fr[0], ring[f % 16]), f
            if f in (n // 4, n - 1):
                marks[f] = (torch.cuda.mem_get_info()[0], rss())
    print(json.dumps(dict(q=marks[n // 4], end=marks[n - 1])))
""")


@pytest.mark.gpu
def test_memory_does_not_grow_with_the_playback(tmp_path):
    """4000 frames of 64 x 96 in batches of a few frames: the free device memory and the host RSS of the child process are the
    same after the first quarter and at the end, up to allocator granularity"""
    import json
    fn = str(tmp_path / "long.lfm")
    env = dict(os.environ, LFM_B200_BATCH_KB="40")
    out = subprocess.run([sys.executable, "-c", _MEM_CHILD, ROOT, fn], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    m = json.loads(out.stdout.strip().splitlines()[-1])
    (free_q, rss_q), (free_end, rss_end) = m["q"], m["end"]
    assert abs(free_q - free_end) <= 2 << 20, m
    assert rss_end - rss_q <= 8 << 20, m


# ---- no device
@pytest.mark.skipif(has_cuda(), reason="checks the no-GPU behaviour")
def test_open_without_a_device_is_code_6(Lhost, oracle, tmp_path):
    a = lf_synth((2, 40, 40), 13)
    fn = str(tmp_path / "o.lfm")
    rc, _ = oracle.write(a, fn, 8, 13, 0)
    assert rc == 0
    r = C.c_void_p(); frames = C.c_uint64(); fb = C.c_uint64()
    assert Lhost.lib.lfmStackReaderOpen(C.byref(r), os.fsencode(fn), None, None, C.byref(frames), C.byref(fb)) == 6 and not r.value
    with pytest.raises(Lhost.LfmError) as ei:
        Lhost.StackReader(fn)
    assert ei.value.code == 6
    # a missing file is found before the device is looked for
    assert Lhost.lib.lfmStackReaderOpen(C.byref(r), os.fsencode(str(tmp_path / "missing.lfm")), None, None, None, None) == 3


def test_reader_argument_checks(Lhost, tmp_path):
    fn = str(tmp_path / "none.lfm")
    with pytest.raises(ValueError):
        Lhost.StackReader(fn, lb=(0, 0, 0, 0, 0))
    with pytest.raises(ValueError):
        Lhost.StackReader(fn, lb=(0, 0, 0), ub=(1, 1, 1))
    with pytest.raises(ValueError):
        Lhost.StackReader(fn, device="cpu")
    assert Lhost.lib.lfmStackReaderOpen(None, os.fsencode(fn), None, None, None, None) == 3
    assert Lhost.lib.lfmStackReaderRead(None, None, 1, None) == 3
    assert Lhost.lib.lfmStackReaderReadDevice(None, None, 1, None) == 3
    assert Lhost.lib.lfmStackReaderClose(None) == 3
