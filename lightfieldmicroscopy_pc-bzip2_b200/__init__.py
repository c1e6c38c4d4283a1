"""lightfieldmicroscopy_pc-bzip2_b200 -- Python (ctypes) binding of the B200-native LFM compression engine.

The product is the C-ABI shared library ``liblfm_b200.so`` built from ``csrc/`` (hand-written sm_100a CUDA kernels +
C++ host layer). This module only loads it and mirrors the reference's C wrapper (``src/klb_Cwrapper.h:40-64``) plus
the extension entry points of ``include/lfm_b200.h`` for tests and the benchmark. There is NO CPU fallback: if the
library is missing the import fails, and every compute call fails with code 6 when no CUDA device is present.

The package directory name contains a hyphen; import it with ``importlib.import_module`` or through the ``lfm_b200``
shim at the repository root.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblfm_b200.so")

UINT16_TYPE = 1
BZIP2 = 1

ERRORS = {0: "ok", 2: "block codec failure", 3: "cannot open / API misuse", 5: "cannot create output / unknown codec",
          6: "CUDA failure", 7: "unsupported"}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError("liblfm_b200.so is not built: run `python __graft_entry__.py` (or "
                          "lightfieldmicroscopy_pc-bzip2_b200/build.py) first; there is no CPU fallback")
    return C.CDLL(LIB_PATH)


lib = _load()

_u32x5 = C.c_uint32 * 5
_f32x5 = C.c_float * 5


class LfmStats(C.Structure):
    _fields_ = [("predictor", C.c_int), ("selected", C.c_int), ("entropy", C.c_float * 8),
                ("ms_select", C.c_double), ("ms_predict", C.c_double), ("ms_rle", C.c_double), ("ms_bwt", C.c_double),
                ("ms_mtf", C.c_double), ("ms_huff", C.c_double), ("ms_decode", C.c_double), ("ms_ibwt", C.c_double),
                ("ms_unrle", C.c_double), ("ms_unpredict", C.c_double), ("ms_h2d", C.c_double), ("ms_d2h", C.c_double),
                ("ms_total", C.c_double), ("gpu_launches", C.c_uint64), ("periodic_blocks", C.c_uint64),
                ("payload_bytes", C.c_uint64), ("ms_imtf", C.c_double)]


# ---- prototypes (include/klb_Cwrapper.h, include/lfm_b200.h)
lib.writeKLBstack.argtypes = [C.c_void_p, C.c_char_p, _u32x5, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
lib.writeKLBstack.restype = C.c_int
lib.writeKLBstackSlices.argtypes = [C.c_void_p, C.c_char_p, _u32x5, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
lib.writeKLBstackSlices.restype = C.c_int
lib.readKLBheader.argtypes = [C.c_char_p, _u32x5, C.POINTER(C.c_int), _f32x5, _u32x5, C.POINTER(C.c_int), C.c_char_p]
lib.readKLBheader.restype = C.c_int
lib.readKLBstack.argtypes = [C.c_char_p, _u32x5, C.POINTER(C.c_int), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
lib.readKLBstack.restype = C.c_void_p
lib.readKLBstackInPlace.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(C.c_int), C.c_int]
lib.readKLBstackInPlace.restype = C.c_int
lib.readKLBroiInPlace.argtypes = [C.c_char_p, C.c_void_p, _u32x5, _u32x5, C.c_int]
lib.readKLBroiInPlace.restype = C.c_int
lib.lfmSetPredictorWay.argtypes = [C.c_int]; lib.lfmSetPredictorWay.restype = C.c_int
lib.lfmGetPredictorWay.restype = C.c_int
lib.lfmSetDevices.argtypes = [C.c_int, C.c_int]; lib.lfmSetDevices.restype = C.c_int
lib.writeLFMstackEx.argtypes = [C.c_void_p, C.c_char_p, _u32x5, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint8, C.c_uint8]
lib.writeLFMstackEx.restype = C.c_int
lib.writeLFMstackDevice.argtypes = lib.writeLFMstackEx.argtypes
lib.writeLFMstackDevice.restype = C.c_int
lib.readLFMroiDevice.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
lib.readLFMroiDevice.restype = C.c_int
lib.readLFMheaderEx.argtypes = [C.c_char_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
lib.readLFMheaderEx.restype = C.c_int
lib.lfmCompressToMemory.argtypes = [C.c_void_p, _u32x5, C.c_void_p, C.c_uint8, C.c_uint8, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
lib.lfmCompressToMemory.restype = C.c_int
lib.lfmCompressToBuffer.argtypes = [C.c_void_p, _u32x5, C.c_void_p, C.c_uint8, C.c_uint8, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
lib.lfmCompressToBuffer.restype = C.c_int
lib.lfmDecompressFromMemory.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p]
lib.lfmDecompressFromMemory.restype = C.c_int
lib.lfmCompressDevice.argtypes = [C.c_void_p, _u32x5, C.c_void_p, C.c_uint8, C.c_uint8, C.POINTER(C.c_uint8), C.c_void_p, C.c_uint64,
                                  C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
lib.lfmCompressDevice.restype = C.c_int
lib.lfmDecompressDevice.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, _u32x5, C.c_void_p, C.c_uint8, C.c_uint8, C.c_void_p]
lib.lfmDecompressDevice.restype = C.c_int
lib.lfmShardCompress.argtypes = [C.c_void_p, _u32x5, C.c_void_p, C.c_uint8, C.c_uint8, C.POINTER(C.c_uint8), C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
lib.lfmShardCompress.restype = C.c_int
lib.lfmShardWritePayload.argtypes = [C.c_char_p, C.c_uint64]; lib.lfmShardWritePayload.restype = C.c_int
lib.lfmShardFetchPayload.argtypes = [C.c_void_p, C.c_uint64]; lib.lfmShardFetchPayload.restype = C.c_int
lib.lfmWriteHeader.argtypes = [C.c_char_p, _u32x5, C.c_void_p, C.c_uint8, C.c_uint8, C.c_void_p, C.c_uint64]; lib.lfmWriteHeader.restype = C.c_int
lib.lfmSelectDevice.argtypes = [C.c_void_p, C.c_uint32 * 2, C.c_uint8, C.POINTER(C.c_int), C.c_void_p]; lib.lfmSelectDevice.restype = C.c_int
lib.lfmNumBlocks.argtypes = [_u32x5, C.c_void_p]; lib.lfmNumBlocks.restype = C.c_uint64
lib.lfmGetLastStats.argtypes = [C.POINTER(LfmStats)]; lib.lfmGetLastStats.restype = C.c_int
lib.lfmLastError.restype = C.c_char_p
lib.lfmDebugEncodeBlock.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
lib.lfmDebugEncodeBlock.restype = C.c_int
lib.lfmDebugPredictDevice.argtypes = [C.c_void_p, C.c_void_p, _u32x5, C.c_uint8, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]
lib.lfmDebugPredictDevice.restype = C.c_int
lib.lfmBz2Compress.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
lib.lfmBz2Compress.restype = C.c_int
lib.lfmBz2CompressDevice.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
lib.lfmBz2CompressDevice.restype = C.c_int
lib.lfmBz2Decompress.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
lib.lfmBz2Decompress.restype = C.c_int
lib.lfmBz2DecompressDevice.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
lib.lfmBz2DecompressDevice.restype = C.c_int
lib.lfmStackWriterOpen.argtypes = [C.POINTER(C.c_void_p), C.c_char_p, _u32x5, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint8, C.c_uint8]
lib.lfmStackWriterOpen.restype = C.c_int
lib.lfmStackWriterAppend.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]; lib.lfmStackWriterAppend.restype = C.c_int
lib.lfmStackWriterAppendDevice.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]; lib.lfmStackWriterAppendDevice.restype = C.c_int
lib.lfmStackWriterClose.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]; lib.lfmStackWriterClose.restype = C.c_int
lib.lfmStackReaderOpen.argtypes = [C.POINTER(C.c_void_p), C.c_char_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
lib.lfmStackReaderOpen.restype = C.c_int
lib.lfmStackReaderRead.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]; lib.lfmStackReaderRead.restype = C.c_int
lib.lfmStackReaderReadDevice.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]; lib.lfmStackReaderReadDevice.restype = C.c_int
lib.lfmStackReaderClose.argtypes = [C.c_void_p]; lib.lfmStackReaderClose.restype = C.c_int

_libc = C.CDLL(None)
_libc.free.argtypes = [C.c_void_p]

EXPORTS = ["writeKLBstack", "writeKLBstackSlices", "readKLBheader", "readKLBstack", "readKLBstackInPlace", "readKLBroiInPlace",
           "lfmSetPredictorWay", "lfmGetPredictorWay", "lfmSetDevices", "writeLFMstackEx", "readLFMheaderEx",
           "lfmCompressToMemory", "lfmCompressToBuffer", "lfmDecompressFromMemory", "lfmCompressDevice", "lfmDecompressDevice", "lfmNumBlocks",
           "lfmGetLastStats", "lfmLastError", "lfmDebugEncodeBlock", "lfmDebugPredictDevice", "lfmDebugParMemcpy",
           "lfmShardCompress", "lfmShardWritePayload", "lfmShardFetchPayload", "lfmWriteHeader", "lfmSelectDevice",
           "lfmBz2Compress", "lfmBz2CompressDevice", "lfmBz2Decompress", "lfmBz2DecompressDevice",
           "writeLFMstackDevice", "readLFMroiDevice",
           "lfmStackWriterOpen", "lfmStackWriterAppend", "lfmStackWriterAppendDevice", "lfmStackWriterClose",
           "lfmStackReaderOpen", "lfmStackReaderRead", "lfmStackReaderReadDevice", "lfmStackReaderClose"]


class LfmError(RuntimeError):
    def __init__(self, code, what):
        msg = lib.lfmLastError()
        super().__init__("%s failed with code %d (%s)%s" % (what, code, ERRORS.get(code, "?"), (": " + msg.decode()) if msg else ""))
        self.code = code


def _xyzct(shape_zyx_or_5):
    """numpy stacks are indexed [t][c][z][y][x]; the library wants x,y,z,c,t"""
    s = list(shape_zyx_or_5)
    while len(s) < 5:
        s.insert(0, 1)
    return _u32x5(s[4], s[3], s[2], s[1], s[0])


def _bs(block_size):
    return None if block_size is None else _u32x5(*block_size)


def set_way(way):
    r = lib.lfmSetPredictorWay(int(way))
    if r < 0:
        raise ValueError("way must be 0 (tiles), 1 (angle) or 2 (space)")
    return r


def set_devices(first=0, count=1):
    return lib.lfmSetDevices(int(first), int(count))


def stats():
    s = LfmStats()
    lib.lfmGetLastStats(C.byref(s))
    return s


def write_stack(img, filename, header_version=0, nnum=13, block_size=None, way=None, codec=BZIP2):
    """img: uint16 array [..., z, y, x]. Mirrors writeKLBstack + the header knobs (writeLFMstackEx).
    img may also be a CUDA torch.uint16 or torch.int16 tensor (uint16 bits, as lf_synth_int makes them) on the first device of
    set_devices: it is compressed where it is (writeLFMstackDevice), into the same file the numpy copy would give."""
    if _is_cuda_tensor(img):
        return _write_stack_device(img, filename, header_version, nnum, block_size, way, codec)
    img = np.ascontiguousarray(img, dtype=np.uint16)
    if way is not None:
        set_way(way)
    bs = _bs(block_size)
    rc = lib.writeLFMstackEx(img.ctypes.data, os.fsencode(filename), _xyzct(img.shape), UINT16_TYPE, -1, None,
                             C.cast(bs, C.c_void_p) if bs is not None else None, codec, None, header_version, nnum)
    if rc:
        raise LfmError(rc, "writeLFMstackEx")
    return rc


class StackWriter:
    """Records a stack frame by frame into `filename` (lfmStackWriterOpen / Append / Close, include/lfm_b200.h).

    shape: [z][y][x] or [t][c][z][y][x] of the whole recording; frames arrive in that order, x fastest.  .append takes a numpy uint16
    array of [n][y][x] or [y][x], or a CUDA torch.uint16 / torch.int16 tensor of the same shapes on the first device of
    set_devices; the frames are copied before it returns.  .close() finishes the file and returns the number of frames kept: all of
    them gives the file write_stack writes for the whole stack, fewer keeps the whole steps of the slowest dimension received.  As a
    context manager the writer is closed on exit, also when the block raises, so that what was recorded is kept.  Errors raise
    LfmError with the library's code."""

    def __init__(self, filename, shape, header_version=0, nnum=13, block_size=None, way=None, codec=BZIP2):
        if len(shape) not in (3, 5):
            raise ValueError("shape is [z][y][x] or [t][c][z][y][x]")
        if way is not None:
            set_way(way)
        self.frame_shape = (int(shape[-2]), int(shape[-1]))
        self._kept = 0
        self._w = C.c_void_p()
        bs = _bs(block_size)
        rc = lib.lfmStackWriterOpen(C.byref(self._w), os.fsencode(filename), _xyzct(shape), UINT16_TYPE, None,
                                    C.cast(bs, C.c_void_p) if bs is not None else None, codec, None, header_version, nnum)
        if rc:
            self._w = None
            raise LfmError(rc, "lfmStackWriterOpen")

    def append(self, frames):
        if self._w is None:
            raise ValueError("the writer is closed")
        if tuple(frames.shape[-2:]) != self.frame_shape or frames.ndim not in (2, 3):
            raise ValueError("append takes [n][y][x] or [y][x] frames of %dx%d pixels" % self.frame_shape)
        n = 1 if frames.ndim == 2 else int(frames.shape[0])
        if _is_cuda_tensor(frames):
            import torch
            if frames.dtype not in (torch.uint16, torch.int16):
                raise TypeError("append takes a torch.uint16 or torch.int16 tensor")
            src = frames.view(torch.int16).contiguous()
            with torch.cuda.device(src.device):
                torch.cuda.current_stream().synchronize()           # the writer copies on its own stream
                rc = lib.lfmStackWriterAppendDevice(self._w, src.data_ptr(), n)
        else:
            if not isinstance(frames, np.ndarray) or frames.dtype != np.uint16:
                raise TypeError("append takes a numpy uint16 array")
            src = np.ascontiguousarray(frames)
            rc = lib.lfmStackWriterAppend(self._w, src.ctypes.data, n)
        if rc:
            raise LfmError(rc, "lfmStackWriterAppend")

    def close(self):
        """finish the file; returns the frames kept"""
        if self._w is None:
            return self._kept
        kept = C.c_uint64()
        rc = lib.lfmStackWriterClose(self._w, C.byref(kept))
        self._w = None
        self._kept = kept.value
        if rc:
            raise LfmError(rc, "lfmStackWriterClose")
        return self._kept

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        if exc[0] is None:
            self.close()
        else:
            try:
                self.close()
            except LfmError:
                pass                                                # the exception of the block is the one to report
        return False

    def __del__(self):
        if getattr(self, "_w", None) is not None:
            try:
                self.close()
            except Exception:
                pass


def read_header(filename):
    xyzct = _u32x5(); ps = _f32x5(); bs = _u32x5(); dt = C.c_int(); ct = C.c_int(); meta = C.create_string_buffer(256)
    rc = lib.readKLBheader(os.fsencode(filename), xyzct, C.byref(dt), ps, bs, C.byref(ct), meta)
    if rc:
        raise LfmError(rc, "readKLBheader")
    hv = C.c_uint8(); nn = C.c_uint8()
    lib.readLFMheaderEx(os.fsencode(filename), C.byref(hv), C.byref(nn))
    return dict(xyzct=list(xyzct), pixelSize=list(ps), blockSize=list(bs), dataType=dt.value, compressionType=ct.value,
                metadata=meta.raw, headerVersion=hv.value, Nnum=nn.value)


def _write_stack_device(img, filename, header_version, nnum, block_size, way, codec):
    import torch
    if img.dtype not in (torch.uint16, torch.int16):
        raise TypeError("write_stack takes a torch.uint16 or torch.int16 tensor")
    src = img.view(torch.int16).contiguous()
    if way is not None:
        set_way(way)
    bs = _bs(block_size)
    with torch.cuda.device(src.device):
        torch.cuda.current_stream().synchronize()               # the engine runs on its own stream
        rc = lib.writeLFMstackDevice(src.data_ptr(), os.fsencode(filename), _xyzct(src.shape), UINT16_TYPE, -1, None,
                                     C.cast(bs, C.c_void_p) if bs is not None else None, codec, None, header_version, nnum)
    if rc:
        raise LfmError(rc, "writeLFMstackDevice")
    return rc


def _device_out(shape, device, out):
    """`out` checked to be a contiguous CUDA tensor of `shape`'s size in bytes on `device` (when given), or a new torch.uint16
    tensor of `shape` on `device`"""
    import torch
    nbytes = 2 * int(np.prod(shape))
    if out is None:
        return torch.empty(shape, dtype=torch.uint16, device=device)
    if not _is_cuda_tensor(out) or not out.is_contiguous() or out.numel() * out.element_size() != nbytes:
        raise ValueError("out= takes a contiguous CUDA tensor of %d bytes" % nbytes)
    if device is not None:
        d = torch.device(device)
        if d.type != "cuda" or (d.index if d.index is not None else torch.cuda.current_device()) != out.device.index:
            raise ValueError("device=%s and out= on %s name different devices" % (device, out.device))
    return out


def _read_device(filename, lb, ub, shape, device, out):
    """decode the box lb..ub (None, None: the whole stack) of a file into a CUDA tensor: `out`, or a new torch.uint16 tensor of
    `shape` on `device`"""
    import torch
    nbytes = 2 * int(np.prod(shape))
    out = _device_out(shape, device, out)
    n = C.c_uint64()
    with torch.cuda.device(out.device):
        torch.cuda.current_stream().synchronize()               # the engine runs on its own stream
        rc = lib.readLFMroiDevice(os.fsencode(filename), lb, ub, out.data_ptr(), nbytes, C.byref(n))
    if rc:
        raise LfmError(rc, "readLFMroiDevice")
    return out


def read_stack(filename, way=None, device=None, out=None):
    """[z][y][x] (c == t == 1) or [t][c][z][y][x] uint16 array of the whole stack.  With `device` (a CUDA device) or `out` (a
    contiguous CUDA tensor of the stack's size in bytes) the stack is decoded into GPU memory instead (readLFMroiDevice) and comes
    back as a torch.uint16 tensor of that shape, or as `out` itself; only the compressed payload crosses PCIe.  Given both,
    `device` must name the device `out` is on (ValueError otherwise)."""
    if way is not None:
        set_way(way)
    h = read_header(filename)
    x, y, z, c, t = h["xyzct"]
    if device is not None or out is not None:
        return _read_device(filename, None, None, (z, y, x) if (c == 1 and t == 1) else (t, c, z, y, x), device, out)
    out = np.empty((t, c, z, y, x), dtype=np.uint16)
    dt = C.c_int()
    rc = lib.readKLBstackInPlace(os.fsencode(filename), out.ctypes.data, C.byref(dt), -1)
    if rc:
        raise LfmError(rc, "readKLBstackInPlace")
    return out.reshape((z, y, x)) if (c == 1 and t == 1) else out


def read_roi(filename, lb, ub, way=None, device=None, out=None):
    """lb/ub: inclusive x,y,z,c,t bounds. Returns array [t][c][z][y][x] of the ROI.  With `device` or `out` as in read_stack, a
    CUDA torch.uint16 tensor of that shape (or `out`)."""
    if way is not None:
        set_way(way)
    shape = [ub[i] - lb[i] + 1 for i in range(5)]
    if device is not None or out is not None:
        return _read_device(filename, _u32x5(*lb), _u32x5(*ub), tuple(shape[::-1]), device, out)
    out = np.empty(shape[::-1], dtype=np.uint16)
    rc = lib.readKLBroiInPlace(os.fsencode(filename), out.ctypes.data, _u32x5(*lb), _u32x5(*ub), -1)
    if rc:
        raise LfmError(rc, "readKLBroiInPlace")
    return out


class StackReader:
    """Plays the box lb..ub (inclusive x,y,z,c,t bounds; None, None: the whole stack) of a .lfm file back frame by frame, in
    bounded memory (lfmStackReaderOpen / Read / ReadDevice / Close, include/lfm_b200.h).  The next batch of frames is decoded on the
    GPU while the caller works on the current one.

    .frames is the number of frames of the box (its z*c*t extent, in [t][c][z] order) and .shape = (frames, y extent, x extent).
    .read(n=1, out=None) returns the next n frames (fewer at the end, none past it) as a numpy uint16 array [n][y][x], or as a CUDA
    torch.uint16 tensor when the reader was opened with device= or `out` (a contiguous CUDA tensor of n frames' bytes, at any even
    byte offset) is given; the rules of read_roi apply.  Iterating yields one frame at a time.  As a context manager the reader is
    closed on exit.  Errors raise LfmError with the library's code."""

    def __init__(self, path, lb=None, ub=None, way=None, device=None):
        if (lb is None) != (ub is None) or (lb is not None and (len(lb) != 5 or len(ub) != 5)):
            raise ValueError("lb and ub are both None or both 5 inclusive x,y,z,c,t bounds")
        if device is not None:
            import torch
            if torch.device(device).type != "cuda":
                raise ValueError("device= names a CUDA device")
        if way is not None:
            set_way(way)
        self._device = device
        self._r = C.c_void_p()
        frames, fb = C.c_uint64(), C.c_uint64()
        rc = lib.lfmStackReaderOpen(C.byref(self._r), os.fsencode(path), _u32x5(*lb) if lb is not None else None,
                                    _u32x5(*ub) if ub is not None else None, C.byref(frames), C.byref(fb))
        if rc:
            self._r = None
            raise LfmError(rc, "lfmStackReaderOpen")
        if lb is None:
            x, y = read_header(path)["xyzct"][:2]
        else:
            x, y = ub[0] - lb[0] + 1, ub[1] - lb[1] + 1
        self.frames = frames.value
        self.shape = (self.frames, int(y), int(x))

    def read(self, n=1, out=None):
        if self._r is None:
            raise ValueError("the reader is closed")
        n = int(n)
        if n < 0:
            raise ValueError("n must be >= 0")
        shape = (n,) + self.shape[1:]
        got = C.c_uint64()
        if self._device is not None or out is not None:
            import torch
            out = _device_out(shape, self._device, out)
            with torch.cuda.device(out.device):
                torch.cuda.current_stream().synchronize()           # the reader copies on its own stream
                rc = lib.lfmStackReaderReadDevice(self._r, out.data_ptr() if n else None, n, C.byref(got))
            if rc:
                raise LfmError(rc, "lfmStackReaderReadDevice")
            return out if got.value == n and out.shape == shape else out.reshape(-1)[:got.value * shape[1] * shape[2]].view(
                (got.value,) + shape[1:])
        a = np.empty(shape, dtype=np.uint16)
        rc = lib.lfmStackReaderRead(self._r, a.ctypes.data, n, C.byref(got))
        if rc:
            raise LfmError(rc, "lfmStackReaderRead")
        return a[:got.value]

    def __iter__(self):
        while True:
            f = self.read(1)
            if len(f) == 0:
                return
            yield f[0]

    def close(self):
        if self._r is None:
            return
        rc = lib.lfmStackReaderClose(self._r)
        self._r = None
        if rc:
            raise LfmError(rc, "lfmStackReaderClose")

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        if exc[0] is None:
            self.close()
        else:
            try:
                self.close()
            except LfmError:
                pass                                                # the exception of the block is the one to report
        return False

    def __del__(self):
        if getattr(self, "_r", None) is not None:
            try:
                self.close()
            except Exception:
                pass


def shard_compress(frames, header_version, nnum=13, block_size=None, way=None):
    """one rank's frames (uint16 [z, y, x], host) -> (stored headerVersion, uint32 size of every local block, payload bytes);
    the streams stay on the rank's GPU until shard_write_payload / shard_fetch_payload (include/lfm_b200.h)"""
    assert frames.dtype == np.uint16 and frames.flags.c_contiguous
    if way is not None:
        set_way(way)
    xyzct = _xyzct(frames.shape)
    bs = _bs(block_size)
    bsp = C.cast(bs, C.c_void_p) if bs is not None else None
    nb = lib.lfmNumBlocks(xyzct, bsp)
    sizes = np.zeros(nb, np.uint32); shv = C.c_uint8(); pb = C.c_uint64()
    rc = lib.lfmShardCompress(frames.ctypes.data, xyzct, bsp, header_version, nnum, C.byref(shv), sizes.ctypes.data, nb, C.byref(pb))
    if rc:
        raise LfmError(rc, "lfmShardCompress")
    return shv.value, sizes, pb.value


def shard_write_payload(filename, file_offset):
    rc = lib.lfmShardWritePayload(os.fsencode(filename), int(file_offset))
    if rc:
        raise LfmError(rc, "lfmShardWritePayload")


def write_header(filename, xyzct, block_size, stored_header_version, nnum, block_offset):
    bo = np.ascontiguousarray(block_offset, dtype=np.uint64)
    bs = _bs(block_size)
    rc = lib.lfmWriteHeader(os.fsencode(filename), _u32x5(*xyzct), C.cast(bs, C.c_void_p) if bs is not None else None,
                            stored_header_version, nnum, bo.ctypes.data, bo.size)
    if rc:
        raise LfmError(rc, "lfmWriteHeader")


def compress_to_bytes(img, header_version=0, nnum=13, block_size=None, way=None):
    img = np.ascontiguousarray(img, dtype=np.uint16)
    if way is not None:
        set_way(way)
    p = C.c_void_p(); n = C.c_uint64()
    bs = _bs(block_size)
    rc = lib.lfmCompressToMemory(img.ctypes.data, _xyzct(img.shape), C.cast(bs, C.c_void_p) if bs is not None else None,
                                 header_version, nnum, C.byref(p), C.byref(n))
    if rc:
        raise LfmError(rc, "lfmCompressToMemory")
    try:
        return C.string_at(p.value, n.value)
    finally:
        _libc.free(p)


def compress_into(img, out, header_version=0, nnum=13, block_size=None, way=None):
    """compress a host stack into the caller's uint8 buffer `out` (numpy array, e.g. a view of pinned memory);
    returns the number of bytes written"""
    assert img.dtype == np.uint16 and img.flags.c_contiguous and out.dtype == np.uint8 and out.flags.c_contiguous
    if way is not None:
        set_way(way)
    n = C.c_uint64()
    bs = _bs(block_size)
    rc = lib.lfmCompressToBuffer(img.ctypes.data, _xyzct(img.shape), C.cast(bs, C.c_void_p) if bs is not None else None,
                                 header_version, nnum, out.ctypes.data, out.nbytes, C.byref(n))
    if rc:
        raise LfmError(rc, "lfmCompressToBuffer")
    return n.value


def decompress_into(data, nbytes, out, way=None):
    """decode the .lfm image held in the uint8 array `data[:nbytes]` into the caller's uint16 array `out`"""
    assert out.dtype == np.uint16 and out.flags.c_contiguous
    if way is not None:
        set_way(way)
    rc = lib.lfmDecompressFromMemory(data.ctypes.data, nbytes, out.ctypes.data)
    if rc:
        raise LfmError(rc, "lfmDecompressFromMemory")
    return out


def decompress_from_bytes(data, shape, way=None):
    if way is not None:
        set_way(way)
    out = np.empty(shape, dtype=np.uint16)
    rc = lib.lfmDecompressFromMemory(data, len(data), out.ctypes.data)
    if rc:
        raise LfmError(rc, "lfmDecompressFromMemory")
    return out


def debug_encode_block(data):
    """Stage-by-stage intermediates of the GPU block encoder for one buffer (even length). Test hook."""
    data = bytes(data)
    n = len(data)
    rle1 = np.zeros(n * 5 // 4 + 64, np.uint8); bwt = np.zeros_like(rle1)
    mtfv = np.zeros(n * 5 // 4 + 64, np.uint16); stream = np.zeros(2 * n + 8400, np.uint8)
    info = (C.c_uint32 * 8)()
    rc = lib.lfmDebugEncodeBlock(data, n, rle1.ctypes.data, bwt.ctypes.data, mtfv.ctypes.data, stream.ctypes.data, info)
    if rc:
        raise LfmError(rc, "lfmDebugEncodeBlock")
    nblock, crc, orig, n_in_use, n_mtf, n_groups, n_sel, sbytes = list(info)
    return dict(nblock=nblock, crc=crc, orig_ptr=orig, n_in_use=n_in_use, n_mtf=n_mtf, n_groups=n_groups, n_sel=n_sel,
                rle1=rle1[:nblock].copy(), bwt=bwt[:nblock].copy(), mtfv=mtfv[:n_mtf].copy(), stream=stream[:sbytes].tobytes())


class _DeviceBytes:
    """an engine-owned device buffer seen by torch through the CUDA array interface (no copy)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def _is_cuda_tensor(data):
    return type(data).__module__.startswith("torch") and getattr(data, "is_cuda", False)


def bz2_compress(data, level=9):
    """One bzip2 stream of `data`, byte-identical to BZ2_bzBuffToBuffCompress(.., level, 0, 30) (include/lfm_b200.h).
    A bytes-like object or numpy array gives `bytes`; a CUDA torch.uint8 tensor (on the first device of set_devices) gives a
    CUDA torch.uint8 tensor."""
    if _is_cuda_tensor(data):
        import torch
        if data.dtype != torch.uint8:
            raise TypeError("bz2_compress takes a torch.uint8 tensor")
        src = data.contiguous().reshape(-1)
        with torch.cuda.device(src.device):
            torch.cuda.current_stream().synchronize()           # the engine runs on its own stream
            p = C.c_void_p(); n = C.c_uint64()
            rc = lib.lfmBz2CompressDevice(src.data_ptr() if src.numel() else None, src.numel(), int(level), C.byref(p), C.byref(n))
            if rc:
                raise LfmError(rc, "lfmBz2CompressDevice")
            return torch.as_tensor(_DeviceBytes(p.value, n.value), device=src.device).clone()
    src = np.ascontiguousarray(np.frombuffer(memoryview(data).cast("B"), np.uint8) if not isinstance(data, np.ndarray)
                               else data.reshape(-1).view(np.uint8))
    n = src.nbytes
    cap = n + n // 64 + 1024 * (n // 99981 + 2) + 4096
    out = np.empty(cap, np.uint8)
    size = C.c_uint64()
    rc = lib.lfmBz2Compress(src.ctypes.data if n else None, n, int(level), out.ctypes.data, cap, C.byref(size))
    if rc == 5:                                                  # cannot happen with the bound above; retry with the size needed
        out = np.empty(size.value, np.uint8)
        rc = lib.lfmBz2Compress(src.ctypes.data if n else None, n, int(level), out.ctypes.data, size.value, C.byref(size))
    if rc:
        raise LfmError(rc, "lfmBz2Compress")
    return out[:size.value].tobytes()


def bz2_decompress(data):
    """Any .bz2 data (one or more concatenated streams, any level) -> the original bytes, CRCs checked (include/lfm_b200.h).
    A bytes-like object or numpy array gives `bytes`; a CUDA torch.uint8 tensor (on the first device of set_devices) gives a CUDA
    torch.uint8 tensor.  The output is sized by one retry when the first guess is too small."""
    size = C.c_uint64()
    if _is_cuda_tensor(data):
        import torch
        if data.dtype != torch.uint8:
            raise TypeError("bz2_decompress takes a torch.uint8 tensor")
        src = data.contiguous().reshape(-1)
        with torch.cuda.device(src.device):
            torch.cuda.current_stream().synchronize()
            out = torch.empty(4 * src.numel() + 4096, dtype=torch.uint8, device=src.device)
            rc = lib.lfmBz2DecompressDevice(src.data_ptr() if src.numel() else None, src.numel(), out.data_ptr(), out.numel(), C.byref(size))
            if rc == 5:
                out = torch.empty(max(1, size.value), dtype=torch.uint8, device=src.device)
                rc = lib.lfmBz2DecompressDevice(src.data_ptr(), src.numel(), out.data_ptr(), out.numel(), C.byref(size))
            if rc:
                raise LfmError(rc, "lfmBz2DecompressDevice")
            return out[:size.value].clone()
    src = np.ascontiguousarray(np.frombuffer(memoryview(data).cast("B"), np.uint8) if not isinstance(data, np.ndarray)
                               else data.reshape(-1).view(np.uint8))
    n = src.nbytes
    out = np.empty(4 * n + 4096, np.uint8)
    rc = lib.lfmBz2Decompress(src.ctypes.data if n else None, n, out.ctypes.data, out.nbytes, C.byref(size))
    if rc == 5:
        out = np.empty(max(1, size.value), np.uint8)
        rc = lib.lfmBz2Decompress(src.ctypes.data, n, out.ctypes.data, out.nbytes, C.byref(size))
    if rc:
        raise LfmError(rc, "lfmBz2Decompress")
    return out[:size.value].tobytes()
