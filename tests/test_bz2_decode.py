"""Reading .bz2 data with lfmBz2Decompress / lfmBz2DecompressDevice / bz2_decompress: any level, concatenated streams, randomised
blocks, false block magics inside Huffman-coded data, and corrupt data."""
import bz2
import ctypes as C
import importlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, has_cuda, lf_synth

BLOCK_MAGIC = 0x314159265359
EOS_MAGIC = 0x177245385090


@pytest.fixture(scope="module")
def L():
    return importlib.import_module("lightfieldmicroscopy_pc-bzip2_b200")


def _code(L, data, cap=None):
    """return code and size of lfmBz2Decompress into a buffer of `cap` bytes"""
    data = bytes(data)
    cap = 4 * len(data) + 4096 if cap is None else cap
    buf = (C.c_uint8 * max(cap, 1))()
    n = C.c_uint64(0)
    return L.lib.lfmBz2Decompress(data, len(data), buf, cap, C.byref(n)), n.value


class BitWriter:
    """MSB-first bit writer, as bzip2 writes its streams"""

    def __init__(self):
        self.bits = []

    def put(self, nbits, v):
        self.bits += [(v >> (nbits - 1 - i)) & 1 for i in range(nbits)]

    def bytes(self):
        b = self.bits + [0] * (-len(self.bits) % 8)
        return np.packbits(np.array(b, np.uint8)).tobytes()


def _crc32_bzip2(data):
    crc = 0xFFFFFFFF
    for byte in data:
        crc ^= byte << 24
        for _ in range(8):
            crc = ((crc << 1) ^ 0x04C11DB7) & 0xFFFFFFFF if crc & 0x80000000 else (crc << 1) & 0xFFFFFFFF
    return crc ^ 0xFFFFFFFF


def _block_text(syms, in_use, orig_ptr):
    """inverse MTF + RUNA/RUNB expansion, inverse BWT by a stable argsort, un-RLE1: the bytes a block of MTF symbols stands for"""
    mtf, last, run, w = list(in_use), [], 0, 1
    for s in syms:
        if s <= 1:
            run += (s + 1) * w; w <<= 1
            continue
        last += [mtf[0]] * run; run, w = 0, 1
        c = mtf.pop(s - 1); mtf.insert(0, c); last.append(c)
    last += [mtf[0]] * run
    L = np.array(last, np.uint8)
    P = np.argsort(L, kind="stable")
    t, text = P[orig_ptr], []
    for _ in range(len(L)):
        text.append(int(L[t])); t = P[t]
    out, i, prev, cnt = [], 0, None, 0
    while i < len(text):
        c = text[i]; i += 1
        out.append(c); cnt = cnt + 1 if c == prev else 1; prev = c
        if cnt == 4 and i < len(text):
            out += [c] * text[i]; i += 1; cnt, prev = 0, None
    return bytes(out)


def _crafted_stream(corrupt_magic=False):
    """the first variant (tail symbols, origPtr) that libbz2 itself accepts: it refuses a block whose text ends on four equal
    bytes without their count byte, which these hand-made blocks do not control"""
    for tail in ([2, 0, 1, 2, 2], [2, 2], [2], [0, 2], [1, 2, 0, 2], [2, 1, 2], [0, 0, 2]):
        for orig in range(4):
            z, text = _crafted_stream_variant(tail, orig, corrupt_magic)
            try:
                ok = bz2.decompress(_crafted_stream_variant(tail, orig, False)[0]) == text
            except OSError:
                ok = False
            if ok:
                return z, text
    raise AssertionError("no crafted variant is valid bzip2")


def _crafted_stream_variant(tail, orig_ptr, corrupt_magic):
    """one block over the bytes 'a', 'b' (alphabet RUNA, RUNB, 2, EOB; code lengths 1, 2, 3, 3: EOB = 111) whose symbols spell the
    48-bit block magic somewhere in the middle -- the magic has no 111, so it parses into RUNA/RUNB/2 codes"""
    codes = {0: (1, 0b0), 1: (2, 0b10), 2: (3, 0b110), 3: (3, 0b111)}
    mbits = [(BLOCK_MAGIC >> (47 - i)) & 1 for i in range(48)]
    inner, i = [], 0
    while i < 48:
        if mbits[i] == 0: inner.append(0); i += 1
        elif mbits[i:i + 2] == [1, 0]: inner.append(1); i += 2
        elif mbits[i:i + 3] == [1, 1, 0]: inner.append(2); i += 3
        else: inner.append(1); i += 2                     # a dangling final 1: RUNB = 10 completes it
    syms = [2, 0, 2, 1] + inner + tail
    in_use = [ord("a"), ord("b")]
    text = _block_text(syms, in_use, orig_ptr)
    crc = _crc32_bzip2(text)
    w = BitWriter()
    for ch in b"BZh9":
        w.put(8, ch)
    w.put(48, BLOCK_MAGIC ^ (1 if corrupt_magic else 0)); w.put(32, crc); w.put(1, 0); w.put(24, orig_ptr)
    w.put(16, 1 << (15 - 6)); w.put(16, (1 << (15 - 1)) | (1 << (15 - 2)))      # bytes 0x61, 0x62
    nsym = len(syms) + 1
    nsel = (nsym + 49) // 50
    w.put(3, 2); w.put(15, nsel)
    for _ in range(nsel):
        w.put(1, 0)                                       # every group uses table 0
    for _ in range(2):                                    # lengths 1, 2, 3, 3 delta coded
        w.put(5, 1); w.put(1, 0); w.put(3, 0b100); w.put(3, 0b100); w.put(1, 0)
    start = len(w.bits)
    for s in syms + [3]:
        w.put(*codes[s])
    body = "".join(map(str, w.bits[start:]))
    assert format(BLOCK_MAGIC, "048b") in body          # the magic is inside the Huffman-coded symbols
    w.put(48, EOS_MAGIC); w.put(32, crc)
    return w.bytes(), text


# ---------------------------------------------------------------------------------------------------- no GPU needed
def test_crafted_stream_is_valid_bzip2():
    z, text = _crafted_stream()
    assert bz2.decompress(z) == text


def test_decode_entry_points_exported_and_check_arguments(L):
    for name in ("lfmBz2Decompress", "lfmBz2DecompressDevice"):
        assert name in L.EXPORTS
    n = C.c_uint64()
    assert L.lib.lfmBz2Decompress(None, 5, None, 0, C.byref(n)) == 3
    assert L.lib.lfmBz2DecompressDevice(None, 5, None, 0, C.byref(n)) == 3
    assert L.lib.lfmBz2Decompress(b"x", 0, None, 0, C.byref(n)) == 2        # as BZ2_bzBuffToBuffDecompress with no input


# ---------------------------------------------------------------------------------------------------- GPU
def _mixed(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.poisson(6, n // 2).astype(np.uint16).tobytes()
    return a[: n // 3] + bytes(5000) + rng.integers(0, 256, n // 3, dtype=np.uint8).tobytes() + a[n // 3:]


@pytest.mark.gpu
def test_decompress_bz2_compress_output_at_every_level(L):
    data = _mixed(1200000, 1)
    for level in range(1, 10):
        assert L.bz2_decompress(bz2.compress(data, level)) == data, level
    st = L.stats()
    assert st.gpu_launches > 0 and st.ms_decode > 0 and st.ms_unrle > 0


@pytest.mark.gpu
def test_decompress_concatenated_streams(L):
    parts = [_mixed(250000 + 1000 * k, 10 + k) for k in range(5)] + [b"", b"q"]
    z = b"".join(bz2.compress(p, lv) for p, lv in zip(parts, (1, 9, 3, 6, 2, 5, 7)))
    assert L.bz2_decompress(z) == b"".join(parts)


@pytest.mark.gpu
@pytest.mark.parametrize("i", [1, 2, 3])
def test_decompress_reference_samples(L, i):
    z = open(os.path.join(GOLDEN, "sample%d.bz2" % i), "rb").read()
    assert L.bz2_decompress(z) == bz2.decompress(z)


@pytest.mark.gpu
def test_decompress_randomised_blocks(L, oracle):
    rng = np.random.default_rng(3)
    for data in (rng.poisson(5, 20000).astype(np.uint16).tobytes(), bytes(5000), rng.integers(0, 256, 300000, dtype=np.uint8).tobytes(),
                 b"ab" * 700, rng.poisson(30, 400000).astype(np.uint16).tobytes()):
        oracle.set_randomised(True)
        try:
            s = oracle.bz2_compress(data, min(9, (len(data) + 99999) // 100000))
        finally:
            oracle.set_randomised(False)
        assert L.bz2_decompress(s) == data


@pytest.mark.gpu
def test_decompress_round_trips_own_streams(L):
    rng = np.random.default_rng(5)
    for data, level in ((lf_synth((3, 512, 700), 13, seed=4).tobytes(), 1), (rng.integers(0, 256, 2500000, dtype=np.uint8).tobytes(), 9),
                        (np.repeat(rng.integers(0, 256, 3000, dtype=np.uint8), rng.integers(1, 600, 3000)).tobytes(), 2), (b"z", 4)):
        assert L.bz2_decompress(L.bz2_compress(data, level)) == data


@pytest.mark.gpu
def test_false_block_magic_inside_huffman_data(L):
    z, text = _crafted_stream()
    assert L.bz2_decompress(z) == text
    assert L.bz2_decompress(z + bz2.compress(b"tail" * 100, 3)) == text + b"tail" * 100
    rc, _ = _code(L, _crafted_stream(corrupt_magic=True)[0])
    assert rc == 2


@pytest.mark.gpu
def test_decompress_rejects_corrupt_data(L):
    data = _mixed(400000, 7)
    z = bz2.compress(data, 2)
    flipped = bytearray(z); flipped[len(z) // 2] ^= 0x08
    bad_level = bytearray(z); bad_level[3] = ord("0")
    big = bytearray(bz2.compress(np.random.default_rng(8).integers(0, 4, 300000, dtype=np.uint8).tobytes(), 9))
    big[3] = ord("1")                                   # its single block holds 300000 bytes: more than level 1 allows
    for name, bad in (("flipped bit", flipped), ("truncated", z[:-7]), ("truncated more", z[: len(z) // 2]),
                      ("trailing garbage", z + b"garbage"), ("level 0", bad_level), ("block over 100000 * level", big),
                      ("no magic", b"BZh9" + bytes(40))):
        assert _code(L, bad)[0] == 2, name
    with pytest.raises(L.LfmError) as e:
        L.bz2_decompress(bytes(flipped))
    assert e.value.code == 2


@pytest.mark.gpu
def test_decompress_too_small_buffer(L):
    data = _mixed(300000, 9)
    z = bz2.compress(data, 5)
    guard = 16
    need = len(data)
    buf = (C.c_uint8 * (need + guard))(*([0x5A] * (need + guard)))
    n = C.c_uint64(0)
    assert L.lib.lfmBz2Decompress(z, len(z), buf, need - 1, C.byref(n)) == 5
    assert n.value == need and bytes(buf) == b"\x5a" * (need + guard)
    assert L.lib.lfmBz2Decompress(z, len(z), buf, need, C.byref(n)) == 0
    assert bytes(buf)[:need] == data and bytes(buf)[need:] == b"\x5a" * guard


@pytest.mark.gpu
def test_decompress_device_and_host_agree(L):
    import torch
    if not has_cuda():
        pytest.skip("no CUDA device")
    data = _mixed(900000, 11)
    z = bz2.compress(data, 1) + bz2.compress(data[:1000], 9)
    t = torch.frombuffer(bytearray(z), dtype=torch.uint8).cuda()
    d = L.bz2_decompress(t)
    assert d.is_cuda and d.dtype == torch.uint8
    assert bytes(d.cpu().numpy()) == L.bz2_decompress(z) == data + data[:1000]
    # a decompressed size above the first guess (4 x the input) takes the retry
    zz = bz2.compress(bytes(3000000), 9)
    assert bytes(L.bz2_decompress(torch.frombuffer(bytearray(zz), dtype=torch.uint8).cuda()).cpu().numpy()) == bytes(3000000)
    assert L.bz2_decompress(zz) == bytes(3000000)
