"""Pin oracle/bz2_oracle.c against the reference's own known-answer vectors and an independent libbz2 (CPU only)."""
import bz2
import ctypes as C
import ctypes.util
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, multiblock_cases


def _cases():
    rng = np.random.default_rng(1)
    return {
        "empty": b"", "one": b"a", "rand30k": rng.integers(0, 256, 30000, dtype=np.uint8).tobytes(),
        "zeros18432": bytes(18432), "zeros1020": bytes(1020), "const300": np.full(73728, 300, np.uint16).tobytes(),
        "const65535": np.full(9216, 65535, np.uint16).tobytes(),
        "poisson147k": rng.poisson(20, 73728).astype(np.uint16).tobytes(),
        "poisson18k": rng.poisson(3, 9216).astype(np.uint16).tobytes(),
        "two_blocks_100k": rng.integers(0, 4, 100000, dtype=np.uint8).tobytes(),
        "runs4": np.repeat(rng.integers(0, 256, 5000, dtype=np.uint8), 4).tobytes(),
        "runs255": np.repeat(rng.integers(0, 256, 100, dtype=np.uint8), 255).tobytes(),
        "runs256": np.repeat(rng.integers(0, 256, 100, dtype=np.uint8), 256).tobytes(),
        "abc": b"abc" * 5000, "ab": b"ab" * 3000,
        "text": open(os.path.join(ROOT, "SURVEY.md"), "rb").read(),
    }


@pytest.mark.parametrize("i,level", [(1, 1), (2, 2), (3, 3)])
def test_reference_known_answer_vectors(oracle, i, level):
    """src/external/bzip2-1.0.6/Makefile:58-69: `bzip2 -1/-2/-3 < sampleN.ref` must equal sampleN.bz2 byte for byte"""
    z = open(os.path.join(GOLDEN, "sample%d.bz2" % i), "rb").read()
    ref = bz2.decompress(z)
    assert oracle.bz2_compress(ref, level) == z
    rc, back = oracle.bz2_decompress(z, len(ref))
    assert rc == 0 and back == ref


@pytest.mark.parametrize("name", sorted(_cases().keys()))
def test_oracle_matches_libbz2(oracle, name):
    data = _cases()[name]
    for level in (1, 2, 9):
        want = bz2.compress(data, level)
        assert oracle.bz2_compress(data, level) == want, (name, level)
        rc, back = oracle.bz2_decompress(want, len(data))
        assert rc == 0 and back == data


def test_oracle_matches_vendored_bzip2_when_built(oracle):
    """BZ2_bzBuffToBuffCompress of the reference's vendored bzip2 1.0.6 (oracle/_ref/libbz2ref.so, oracle/build_ref.py), or of the
    system's libbz2 when oracle/_ref is not built"""
    ref = _vendored_bz2()
    if ref is None:
        pytest.skip("neither oracle/_ref/libbz2ref.so nor a libbz2 that ctypes.util.find_library('bz2') finds and loads")
    for name, data in _cases().items():
        for level in (1, 2):
            assert oracle.bz2_compress(data, level) == ref(data, level), (name, level)


def test_decoder_rejects_corruption(oracle):
    data = np.random.default_rng(5).poisson(9, 5000).astype(np.uint16).tobytes()
    z = bytearray(bz2.compress(data, 1))
    z[len(z) // 2] ^= 0x10
    rc, _ = oracle.bz2_decompress(bytes(z), len(data))
    assert rc != 0
    assert oracle.bz2_decompress(b"BZx9", 10)[0] == -1


def test_trace_is_consistent(oracle):
    data = np.random.default_rng(2).poisson(5, 9216).astype(np.uint16).tobytes()
    out, blocks = oracle.bz2_compress(data, 1, trace=True)
    assert out == bz2.compress(data, 1) and len(blocks) == 1
    b = blocks[0]
    assert b["mtfv"][-1] == b["n_in_use"] + 1 and len(b["bwt"]) == b["nblock"]
    # the BWT column is a permutation of the block
    assert np.array_equal(np.sort(b["bwt"]), np.sort(b["rle1"]))


def _vendored_bz2():
    """BZ2_bzBuffToBuffCompress of oracle/_ref/libbz2ref.so; without it, of the system's libbz2 (the one Python's bz2 module links):
    the compressor's output has not changed since the vendored 1.0.6"""
    so = os.path.join(ROOT, "oracle", "_ref", "libbz2ref.so")
    if not os.path.exists(so):
        so = ctypes.util.find_library("bz2")
        if so is None:
            return None
    try:
        ref = C.CDLL(so)
    except OSError:
        return None
    ref.BZ2_bzBuffToBuffCompress.argtypes = [C.c_char_p, C.POINTER(C.c_uint), C.c_char_p, C.c_uint, C.c_int, C.c_int, C.c_int]
    def compress(data, level):
        cap = C.c_uint(len(data) * 2 + 1000); buf = C.create_string_buffer(cap.value)
        assert ref.BZ2_bzBuffToBuffCompress(buf, C.byref(cap), data, len(data), level, 0, 30) == 0
        return buf.raw[:cap.value]
    return compress


# Python's bz2.compress drives libbz2 with BZ_RUN and then BZ_FINISH; the reference calls BZ2_bzBuffToBuffCompress, which enters
# BZ_FINISH at once.  The two differ in exactly one situation: the LAST input byte is the one that fills a block.  In finishing mode
# that byte is flushed into the full block (handle_compress: avail_in_expect == 0 is tested before nblock >= nblockMAX), in running
# mode the block is closed first and the byte opens a new one.  The oracle follows the reference (BuffToBuff).
STREAMING_DIFFERS = {"l2_exact_plus1"}


@pytest.mark.parametrize("name", sorted(multiblock_cases().keys()))
def test_oracle_multi_block_streams(oracle, name):
    """streams of several bzip2 blocks and the block-closing rules, at the level klb_imageIO.cpp:108 picks for the size:
    against BZ2_bzBuffToBuffCompress (_vendored_bz2) and against libbz2's streaming API"""
    data = multiblock_cases()[name]
    level = min(9, (len(data) + 99999) // 100000)
    got, blocks = oracle.bz2_compress(data, level, trace=True)
    ref = _vendored_bz2()
    if ref is not None:
        assert got == ref(data, level), "vendored bzip2 1.0.6, BZ2_bzBuffToBuffCompress"
    if name not in STREAMING_DIFFERS:
        assert got == bz2.compress(data, level)
    elif ref is None:
        pytest.skip("this case is only pinned by BZ2_bzBuffToBuffCompress (neither oracle/_ref/libbz2ref.so nor a libbz2 that "
                    "ctypes.util.find_library('bz2') finds and loads)")
    expect_blocks = {"l2_exact_plus1": 1, "l2_exact_plus3": 2, "l2_tail_run2": 2, "l2_run4_across": 2, "l2_runs4": 2,
                     "l1_poisson": 1, "l1_random_2blocks": 2, "l9_2MB_3blocks": 3, "l9_1MB_runs": 2}
    if name in expect_blocks:
        assert len(blocks) == expect_blocks[name]
    assert bz2.decompress(got) == data
    rc, back = oracle.bz2_decompress(got, len(data))
    assert rc == 0 and back == data


def test_randomised_blocks_are_pinned_to_libbz2(oracle):
    """bzip2 <= 0.9.0 could set the "randomised" bit of a block (BZ_RAND_*, randtable.c); the oracle's test hook writes such
    streams: libbz2 itself must decode them back to the input (that pins the mask positions), and so must the oracle's decoder"""
    rng = np.random.default_rng(3)
    cases = [rng.poisson(5, 20000).astype(np.uint16).tobytes(), bytes(5000), rng.integers(0, 256, 300000, dtype=np.uint8).tobytes(),
             b"ab" * 700, rng.poisson(30, 400000).astype(np.uint16).tobytes()]
    for data in cases:
        level = min(9, (len(data) + 99999) // 100000)
        oracle.set_randomised(True)
        try:
            s = oracle.bz2_compress(data, level)
        finally:
            oracle.set_randomised(False)
        assert s != oracle.bz2_compress(data, level)
        assert bz2.decompress(s) == data
        rc, back = oracle.bz2_decompress(s, len(data) + 16)
        assert rc == 0 and back == data
