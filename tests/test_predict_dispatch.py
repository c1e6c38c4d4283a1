"""Every forward and inverse predictor kernel that launch_predict_fwd / launch_unpredict (csrc/lfm_predict.cu) can choose,
run at a shape that chooses it and checked against the oracle's plain C statement of the prediction rules.

A row of ROWS names a stack (frames x H x W, Nnum), a way, its predictors, image and / or video mode, the byte offsets of
the device buffers (views into a larger tensor) and the run-time switches it needs.  For each row, through
lfmDebugPredictDevice:
  * forward: the GPU's symbols equal oracle.predict_frame for every frame (odd video frames: prev = the frame before);
  * inverse: from the ORACLE's symbols, into a buffer filled with a sentinel, the GPU gives the stack back exactly, and so
    does oracle.unpredict_frame;
  * the bytes around both buffer views are untouched;
  * torch.profiler (CUDA activities) lists the kernel the row is there for, and for a fall-back row not the kernel the
    dispatcher prefers.
Stacks of more than 65535 frames repeat a few distinct frames with a period that does not divide 65536, so every frame is
checked while the oracle only predicts one period; a kernel that reads the wrong frame index still fails.

The switches are read once per process, on first use.  So every group of rows with the same switches runs in a fresh
child process, from which every inherited LFM_B200_* variable is removed: a setting left behind by an earlier test in the
same process cannot change which kernel a row reaches.
"""
import ctypes as C
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from conftest import Oracle, lf_synth

BIG = 1 << 16                    # frame counts from here on are stored as repeats of PERIOD distinct frames
PERIOD = 7                       # 65536 % 7 != 0 and 65536 % 14 != 0 (video pairs)
SENTINEL = -21555                # 0xABCD


class Row:
    def __init__(self, name, way, ks, shape, T, video=(0,), off=(0, 0), env=None, fwd=(), not_fwd=(), inv=(), not_inv=()):
        self.name, self.way, self.ks, self.shape, self.T, self.video = name, way, tuple(ks), shape, T, tuple(video)
        self.off = off                  # byte offsets of the source and the destination view of each call
        self.env = dict(env or {})
        # fwd / inv: kernels that must run in the capture of EVERY (predictor, video mode) of the row -- an entry (pattern, ks)
        # only for those predictors; not_fwd / not_inv: kernels that must run in none of them
        self.fwd, self.not_fwd, self.inv, self.not_inv = fwd, not_fwd, inv, not_inv

    def expected(self, pats):
        """(pattern, predictors it is expected for)"""
        return [(p, self.ks) if isinstance(p, str) else (p[0], tuple(p[1])) for p in pats]

    @property
    def group(self):
        return ",".join("%s=%s" % kv for kv in sorted(self.env.items())) or "default"


K7, K_NOT2, K_SCAN, K_NOSCAN = range(1, 8), (1, 3, 4, 5, 6, 7), (1, 2, 4), (3, 5, 6, 7)
FWD2, FWD, FWD_ROWS = "k_predict_fwd2<", "k_predict_fwd<", "k_predict_fwd_rows<"
SEG, COLS4, COLS2, COLS1, UROWS = "k_unscan_cols_seg", "k_unscan_cols<false, 4>", "k_unscan_cols<false, 2>", "k_unscan_cols<false, 1>", "k_unscan_rows<"
GRID2, GRID1, SPACE, ANGLE, TANGLE = "k_unpredict_grid<2,", "k_unpredict_grid<1,", "k_unpredict_space(", "k_unpredict_angle(", "k_unpredict_tiles_angle<"
BANDS, CLUSTER, ROW0, UCOLS2, STRIPS = "k_unpredict_bands<", "k_unpredict(", "k_unpredict_row0<", "k_unpredict_cols2<", "k_unpredict_strips<"

ROWS = [
    # ---- forward kernels
    Row("fwd2_w8_h_lt_nnum", 0, K7, (4, 7, 8), 11, video=(0, 1), fwd=(FWD2,)),
    Row("fwd2_w8_angle_space", 1, K7, (3, 7, 8), 11, fwd=(FWD2,)),
    Row("fwd2_space_w8", 2, K7, (3, 7, 8), 11, fwd=(FWD2,)),
    Row("fwd_odd_w", 0, K7, (3, 40, 57), 11, video=(0, 1), fwd=(FWD,), not_fwd=(FWD2,)),
    Row("fwd_odd_w_angle", 1, K7, (3, 40, 57), 11, fwd=(FWD,), not_fwd=(FWD2,)),
    Row("fwd_w64_off2", 2, K7, (3, 40, 64), 11, off=(2, 2), fwd=(FWD,), not_fwd=(FWD2,)),
    Row("fwd_w64_sym_off2", 0, K7, (3, 40, 64), 11, video=(0, 1), off=(0, 2), fwd=(FWD,), not_fwd=(FWD2,)),
    # Nnum 121..127: the tile kernel with its widest halo (128 columns, half the tile); from Nnum 128 on: the row kernel
    Row("fwd_halo128_nnum121_tiles", 0, K7, (2, 300, 260), 121, video=(0, 1), fwd=(FWD,), not_fwd=(FWD_ROWS, FWD2)),
    Row("fwd_halo128_nnum127_angle", 1, K7, (2, 300, 260), 127, fwd=(FWD,), not_fwd=(FWD_ROWS, FWD2)),
    Row("fwd_rows_nnum128_tiles", 0, K7, (2, 300, 260), 128, video=(0, 1), fwd=(FWD_ROWS,), not_fwd=(FWD, FWD2)),
    Row("fwd_rows_nnum128_angle", 1, K7, (2, 300, 260), 128, fwd=(FWD_ROWS,), not_fwd=(FWD, FWD2)),
    Row("fwd_rows_nnum128_space", 2, K7, (2, 300, 260), 128, fwd=(FWD_ROWS,), not_fwd=(FWD, FWD2)),
    Row("fwd_rows_nnum255_tiles", 0, K7, (2, 270, 300), 255, video=(0, 1), fwd=(FWD_ROWS,)),
    Row("fwd_rows_nnum255_angle", 1, K7, (2, 270, 300), 255, fwd=(FWD_ROWS,)),
    Row("fwd_rows_nnum255_space", 2, K7, (2, 270, 300), 255, fwd=(FWD_ROWS,)),
    Row("nnum1_tiles", 0, K7, (3, 20, 24), 1, video=(0, 1)),
    Row("nnum1_angle", 1, K7, (3, 20, 24), 1),
    Row("nnum1_space", 2, K7, (3, 20, 24), 1),
    Row("nnum2_tiles", 0, K7, (3, 21, 23), 2, video=(0, 1)),
    Row("nnum2_angle", 1, K7, (3, 21, 23), 2),
    Row("nnum2_space", 2, K7, (3, 21, 23), 2),
    Row("w_lt_nnum_tiles", 0, K7, (3, 9, 3), 5, video=(0, 1)),
    Row("w_lt_nnum_angle", 1, K7, (3, 9, 3), 5),
    Row("w_lt_nnum_space", 2, K7, (3, 9, 3), 5),
    Row("h1_tiles", 0, K7, (4, 1, 40), 5, video=(0, 1)),
    Row("h1_angle", 1, K7, (4, 1, 40), 5),
    Row("h1_space", 2, K7, (4, 1, 40), 5),
    Row("w1_tiles", 0, K7, (4, 30, 1), 5, video=(0, 1)),
    Row("w1_angle", 1, K7, (4, 30, 1), 5),
    Row("w1_space", 2, K7, (4, 30, 1), 5),
    # ---- way space inverse: prefix-sum passes (predictors 1, 2, 4)
    # (predictor 1 has no full-width column pass: only the first tile column, always one pixel wide)
    Row("scan_cols_seg", 2, K_SCAN, (2, 60, 64), 11, inv=((SEG, (2, 4)), UROWS), not_inv=(COLS4, COLS2)),
    Row("scan_cols2_w66", 2, K_SCAN, (2, 60, 66), 11, inv=((COLS2, (2, 4)), UROWS), not_inv=(SEG, COLS4)),
    Row("scan_cols2_off4", 2, K_SCAN, (2, 60, 64), 11, off=(4, 4), inv=((COLS2, (2, 4)), UROWS), not_inv=(SEG, COLS4)),
    Row("scan_cols1_w67", 2, K_SCAN, (2, 60, 67), 11, inv=(COLS1, UROWS), not_inv=(SEG, COLS4, COLS2)),
    Row("scan_cols1_off2", 2, K_SCAN, (2, 60, 64), 11, off=(2, 2), inv=(COLS1, UROWS), not_inv=(SEG, COLS4, COLS2)),
    Row("scan_rows_r1_short_frame", 2, K_SCAN, (1, 30, 64), 11, inv=(UROWS,)),
    Row("scan_rows_r8", 2, K_SCAN, (80, 64, 64), 11, inv=(UROWS, (SEG, (2, 4)))),
    Row("scan_l2_groups", 2, (4,), (9, 2048, 2048), 15, inv=(UROWS, SEG)),
    # ---- way space inverse: sub-aperture grid (G sub-images per CTA) and the fall-back beyond shared memory
    Row("grid2_g4", 2, K_NOSCAN, (2, 1024, 1024), 7, inv=(GRID2,), not_inv=(SPACE,)),
    Row("grid2_g3", 2, K_NOSCAN, (1, 1024, 1024), 6, inv=(GRID2,), not_inv=(SPACE,)),
    Row("grid2_g2", 2, K_NOSCAN, (1, 1024, 1024), 5, inv=(GRID2,), not_inv=(SPACE,)),
    Row("grid2_g1", 2, K_NOSCAN, (1, 1024, 1024), 4, inv=(GRID2,), not_inv=(SPACE,)),
    Row("space_1024_nnum3", 2, K7, (1, 1024, 1024), 3, inv=((SPACE, K_NOSCAN), (UROWS, K_SCAN)), not_inv=(GRID2,)),
    Row("space_w24600", 2, K_SCAN, (1, 40, 24600), 15, inv=(SPACE,), not_inv=(GRID2, UROWS, SEG, COLS4, COLS2, COLS1)),
    # ---- way angle inverse
    Row("angle_tiles_nnum28", 1, K_NOT2, (2, 100, 168), 28, inv=(GRID1, TANGLE), not_inv=(ANGLE,)),
    Row("angle_tiles_nnum28_odd_w", 1, K_NOT2, (2, 90, 150), 28, inv=(GRID1, TANGLE), not_inv=(ANGLE,)),
    Row("angle_nnum29", 1, K_NOT2, (2, 100, 150), 29, inv=(ANGLE,), not_inv=(TANGLE,)),
    Row("angle_1024_nnum3", 1, K_NOT2, (1, 1024, 1024), 3, inv=(ANGLE,), not_inv=(TANGLE, GRID1)),
    # ---- way tiles inverse
    Row("bands_nnum30_odd", 0, K_NOT2, (7, 70, 100), 30, video=(0, 1), inv=(BANDS,), not_inv=(CLUSTER,)),
    Row("bands_nnum30_even", 0, K_NOT2, (8, 70, 100), 30, video=(0, 1), inv=(BANDS,), not_inv=(CLUSTER,)),
    Row("cluster_nnum31", 0, K_NOT2, (4, 70, 100), 31, inv=(CLUSTER,), not_inv=(BANDS,)),
    Row("cols2_tiles", 0, (2,), (5, 60, 100), 13, video=(0, 1), inv=(ROW0, UCOLS2), not_inv=(CLUSTER, STRIPS)),
    Row("cols2_angle", 1, (2,), (5, 60, 100), 13, inv=(ROW0, UCOLS2), not_inv=(CLUSTER, STRIPS)),
    Row("strips_h1_tiles", 0, (2,), (130, 1, 200), 13, inv=(STRIPS,), not_inv=(CLUSTER, UCOLS2)),
    Row("strips_h1_angle", 1, (2,), (130, 1, 200), 13, inv=(STRIPS,), not_inv=(CLUSTER, UCOLS2)),
    Row("strips_h1_video", 0, (2,), (260, 1, 200), 13, video=(1,), inv=(STRIPS,), not_inv=(CLUSTER, UCOLS2)),
    Row("cluster_1_frame_csz1", 0, K_NOT2, (1, 40, 50), 13, video=(0, 1), inv=(CLUSTER,), not_inv=(BANDS,)),
    Row("cluster_2_frames_csz8", 0, K_NOT2, (2, 1024, 1024), 13, video=(0, 1), inv=(CLUSTER,), not_inv=(BANDS,)),
    Row("cluster_rows_k2_nnum33", 0, (2,), (3, 100, 136), 33, video=(0, 1), inv=(CLUSTER,), not_inv=(UCOLS2, STRIPS)),
    Row("cluster_rows_k2_nnum33_angle", 1, (2,), (3, 100, 136), 33, inv=(CLUSTER,), not_inv=(UCOLS2, STRIPS)),
    # ---- more frames than one grid dimension holds
    Row("frames65537_tiles", 0, K7, (65537, 16, 16), 5, fwd=(FWD2,), inv=((BANDS, K_NOT2), (ROW0, (2,)), (UCOLS2, (2,)))),
    Row("frames65537_angle", 1, K7, (65537, 16, 16), 5, fwd=(FWD2,), inv=((GRID1, K_NOT2), (TANGLE, K_NOT2), (UCOLS2, (2,)))),
    Row("frames65537_space", 2, K7, (65537, 16, 16), 5, fwd=(FWD2,), inv=((UROWS, K_SCAN), (GRID2, K_NOSCAN))),
    Row("frames131074_video", 0, K7, (131074, 8, 16), 5, video=(1,), fwd=(FWD2,), inv=((BANDS, K_NOT2), (UCOLS2, (2,)))),
    # ---- rows that need a switch (child process of their own)
    Row("tma_off_cp_async", 0, K7, (3, 40, 64), 11, video=(0, 1), env={"LFM_B200_TMA": "0"}, fwd=(FWD2,)),
    Row("tma_off_cp_async_space", 2, K7, (3, 40, 64), 11, env={"LFM_B200_TMA": "0"}, fwd=(FWD2,)),
    Row("scan_seg_off_cols4", 2, K_SCAN, (2, 60, 64), 11, env={"LFM_B200_SCAN_SEG": "0"}, inv=((COLS4, (2, 4)), UROWS), not_inv=(SEG,)),
    Row("scans_off_grid", 2, K_SCAN, (2, 60, 64), 11, env={"LFM_B200_SCANS": "0"}, inv=(GRID2,), not_inv=(UROWS, SEG)),
    Row("bands_r1", 0, K_NOT2, (7, 70, 100), 13, video=(0, 1), env={"LFM_B200_BANDS_R": "1"}, inv=(BANDS,), not_inv=(CLUSTER,)),
]
_STRIPS_ENV = {"LFM_B200_BANDS": "0", "LFM_B200_COLS": "0", "LFM_B200_STRIPS_MIN": "1"}
for _shape, _off, _tag in (((6, 40, 64), (0, 0), "w64"), ((6, 40, 67), (0, 0), "w67"), ((6, 40, 64), (2, 2), "w64_off2")):
    ROWS.append(Row("strips_all_tiles_" + _tag, 0, K7, _shape, 13, video=(0, 1), off=_off, env=_STRIPS_ENV,
                    inv=(STRIPS,), not_inv=(BANDS, UCOLS2, CLUSTER)))
    ROWS.append(Row("strips_all_angle_k2_" + _tag, 1, (2,), _shape, 13, off=_off, env=_STRIPS_ENV,
                    inv=(STRIPS,), not_inv=(UCOLS2, CLUSTER)))
BY_NAME = {r.name: r for r in ROWS}
assert len(BY_NAME) == len(ROWS)


# ------------------------------------------------------------------------------------------------ data and oracle
def base_frames(row):
    """the distinct frames of a row's stack: all of them, or PERIOD of them for stacks of BIG frames and more"""
    F, H, W = row.shape
    n = F if F < BIG else PERIOD
    rng = np.random.default_rng([F, H, W, row.T])
    out = np.empty((n, H, W), np.uint16)
    for z in range(n):
        f = lf_synth((1, H, W), row.T, seed=1000 + z)[0].astype(np.int64) + rng.integers(0, 400, (H, W))
        wild = rng.random((H, W)) < 0.03                               # full-range pixels: residuals wrap around int16
        f[wild] = rng.integers(0, 65536, int(wild.sum()))
        out[z] = np.clip(f, 0, 65535)
    return out


def sym_period(row, video):
    """frames of the stack whose symbols the oracle computes; symbols of frame z are those of frame z % period"""
    F = row.shape[0]
    if F < BIG:
        return F
    return 2 * PERIOD if video else PERIOD


def unpredict_frame(oracle, sym, prev, T, way, k, zflag):
    """oracle.lfmo_unpredict_frame: symbols -> pixels, in raster order"""
    sym = np.ascontiguousarray(sym, np.uint16); H, W = sym.shape
    prev_p = np.ascontiguousarray(prev, np.uint16).ctypes.data if prev is not None else None
    out = np.empty((H, W), np.uint16)
    assert oracle.lib.lfmo_unpredict_frame(sym.ctypes.data, prev_p, out.ctypes.data, W, H, T, way, k, zflag) == 0
    return out


def oracle_symbols(oracle, row, base, k, video):
    n = sym_period(row, video)
    P = base.shape[0]
    out = np.empty((n,) + base.shape[1:], np.uint16)
    for z in range(n):
        zf = video & z & 1
        out[z] = oracle.predict_frame(base[z % P], base[(z - 1) % P] if zf else None, row.T, row.way, k, zf)
    return out


def combos(row):
    return [(k, v) for v in row.video for k in row.ks]


# ------------------------------------------------------------------------------------------------ oracle self-consistency
@pytest.mark.parametrize("name", [r.name for r in ROWS])
def test_oracle_round_trip(oracle, name):
    """unpredict_frame(predict_frame(x)) == x at every row's shape, way, predictor and video mode (no GPU needed): the
    reference the GPU rows are held to is itself consistent"""
    row = BY_NAME[name]
    base = base_frames(row)
    P, H, W = base.shape
    nz = P if P * H * W <= 2_000_000 else 2                         # large frames: one even and one odd frame
    for k, video in combos(row):
        for z in range(min(nz, sym_period(row, video))):
            zf = video & z & 1
            prev = base[(z - 1) % P] if zf else None
            s = oracle.predict_frame(base[z % P], prev, row.T, row.way, k, zf)
            back = unpredict_frame(oracle, s, prev, row.T, row.way, k, zf)
            assert np.array_equal(back, base[z % P]), (name, k, video, z)


def test_rows_cover_every_switch_and_kernel():
    """the table names every kernel of the dispatcher at least once (a kernel name typo would make a row vacuous)"""
    named = {p for r in ROWS for p, _ in r.expected(r.fwd + r.inv)}
    for p in (FWD2, FWD, FWD_ROWS, SEG, COLS4, COLS2, COLS1, UROWS, GRID2, GRID1, SPACE, ANGLE, TANGLE, BANDS, CLUSTER, ROW0,
              UCOLS2, STRIPS):
        assert p in named, p


# ------------------------------------------------------------------------------------------------ GPU rows (child side)
def _kernels(prof):
    return sorted({e.key for e in prof.key_averages() if "lfm::" in e.key})


def _ran(names, pat):
    return any(pat in n for n in names)


def _views(torch, n, off_bytes, fill):
    """a view of n int16 at off_bytes past a 16-byte boundary of a larger buffer filled with `fill`"""
    assert off_bytes % 2 == 0
    lead = 8 + off_bytes // 2
    backing = torch.full((n + lead + 8,), fill, dtype=torch.int16, device="cuda")
    return backing, backing[lead:lead + n], lead


def _margins_intact(backing, lead, n, fill):
    return bool((backing[:lead] == fill).all()) and bool((backing[lead + n:] == fill).all())


def _first_diff(got, want):
    bad = (got != want).nonzero()
    return tuple(int(i) for i in bad[0]) if bad.numel() else None


def run_row(L, oracle, row):
    """all checks of one row; returns dict(errors=[...], fwd_kernels={"k,video": [...]}, inv_kernels={...})"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    F, H, W = row.shape
    n = F * H * W
    base = base_frames(row)
    P = base.shape[0]
    idx = torch.arange(F, device="cuda")
    stack = torch.from_numpy(base.view(np.int16)).cuda()[idx % P].reshape(-1)
    xyz = L._u32x5(W, H, F, 1, 1)
    ms = C.c_float()
    errors = []
    L.set_way(row.way)
    fwd_names, inv_names = {}, {}
    for k, video in combos(row):
        tag = "k=%d video=%d" % (k, video)
        osym = oracle_symbols(oracle, row, base, k, video)
        Q = osym.shape[0]
        want_sym = torch.from_numpy(osym.view(np.int16)).cuda()[idx % Q].reshape(-1)
        # forward: the stack -> symbols
        bi, src, li = _views(torch, n, row.off[0], 0)
        src.copy_(stack)
        bo, dst, lo = _views(torch, n, row.off[1], SENTINEL)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            rc = L.lib.lfmDebugPredictDevice(src.data_ptr(), dst.data_ptr(), xyz, row.T, k, video, 0, 1, C.byref(ms))
            torch.cuda.synchronize()
        fwd_names["%d,%d" % (k, video)] = _kernels(prof)
        if rc:
            errors.append("%s forward: code %d (%s)" % (tag, rc, L.lib.lfmLastError().decode()))
            continue
        if not torch.equal(dst, want_sym):
            at = _first_diff(dst.view(F, H, W), want_sym.view(F, H, W))
            errors.append("%s forward: symbols differ from the oracle's, first at (z, y, x) = %s" % (tag, at))
        if not _margins_intact(bo, lo, n, SENTINEL) or not _margins_intact(bi, li, n, 0) or not torch.equal(src, stack):
            errors.append("%s forward: wrote outside its output view" % tag)
        # inverse: the oracle's symbols -> the stack
        bi, src, li = _views(torch, n, row.off[0], 0)
        src.copy_(want_sym)
        bo, dst, lo = _views(torch, n, row.off[1], SENTINEL)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            rc = L.lib.lfmDebugPredictDevice(src.data_ptr(), dst.data_ptr(), xyz, row.T, k, video, 1, 1, C.byref(ms))
            torch.cuda.synchronize()
        inv_names["%d,%d" % (k, video)] = _kernels(prof)
        if rc:
            errors.append("%s inverse: code %d (%s)" % (tag, rc, L.lib.lfmLastError().decode()))
            continue
        if not torch.equal(dst, stack):
            at = _first_diff(dst.view(F, H, W), stack.view(F, H, W))
            errors.append("%s inverse: pixels differ from the stack, first at (z, y, x) = %s" % (tag, at))
        if not _margins_intact(bo, lo, n, SENTINEL) or not _margins_intact(bi, li, n, 0) or not torch.equal(src, want_sym):
            errors.append("%s inverse: wrote outside its output view" % tag)
        for z in range(min(2, Q)):                                     # the oracle's own inverse of its symbols
            zf = video & z & 1
            if not np.array_equal(unpredict_frame(oracle, osym[z], base[(z - 1) % P] if zf else None, row.T, row.way, k, zf), base[z % P]):
                errors.append("%s oracle: unpredict_frame(predict_frame) != frame %d" % (tag, z))
    return dict(errors=errors, fwd_kernels=fwd_names, inv_kernels=inv_names)


SELECT_FRAMES = {
    # name: (frame maker, Nnum, ways)
    "7x9": (lambda: np.random.default_rng(1).poisson(50, (7, 9)).astype(np.uint16), 3, (0, 1, 2)),
    "37x53": (lambda: lf_synth((1, 37, 53), 5, seed=2)[0], 5, (0, 1, 2)),
    "2048x2048": (lambda: lf_synth((1, 2048, 2048), 15, seed=3)[0], 15, (0, 2)),
    "1000x1001": (lambda: lf_synth((1, 1000, 1001), 13, seed=4)[0], 13, (1,)),
    "const": (lambda: np.full((64, 64), 1234, np.uint16), 13, (0, 1, 2)),
}


def run_select(L):
    out = {}
    for name, (make, T, ways) in SELECT_FRAMES.items():
        f = make()
        for way in ways:
            L.compress_to_bytes(f[None], header_version=0, nnum=T, way=way)
            st = L.stats()
            out["%s/way%d" % (name, way)] = dict(selected=st.selected, predictor=st.predictor,
                                                 bits=[struct.unpack("<I", struct.pack("<f", e))[0] for e in st.entropy])
    return out


def child_main(argv):
    """python test_predict_dispatch.py rows NAME... | select: run in this (fresh) process, print one RESULT line of JSON"""
    import lfm_b200 as L
    L.set_devices(0, 1)
    if argv[0] == "select":
        res = run_select(L)
    else:
        oracle = Oracle()
        res = {}
        for name in argv[1:]:
            try:
                res[name] = run_row(L, oracle, BY_NAME[name])
            except Exception as e:                                      # report, and go on with the next row
                res[name] = dict(errors=["%s: %s" % (type(e).__name__, e)], fwd_kernels={}, inv_kernels={})
    print("RESULT " + json.dumps(res), flush=True)


# ------------------------------------------------------------------------------------------------ GPU rows (pytest side)
_results = {}        # key -> the child's result, or the text of its failure: each child runs at most once per session


def _child(args, env_extra, timeout):
    env = {k: v for k, v in os.environ.items() if not k.startswith("LFM_B200_")}
    env.update(env_extra)
    env["LFM_B200_DEBUG_POISON"] = "1"
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__)] + list(args)
    try:
        p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return "child %s did not finish in %d s" % (args[:1], timeout)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")]
    if p.returncode != 0 or not lines:
        return "child %s failed (exit %d):\n%s\n%s" % (args[:1], p.returncode, p.stdout[-3000:], p.stderr[-3000:])
    return json.loads(lines[-1][len("RESULT "):])


def _cached_child(key, args, env_extra, timeout):
    """the child's result; a child that failed is not started again, every later test of its group reports that failure"""
    if key not in _results:
        _results[key] = _child(args, env_extra, timeout)
    res = _results[key]
    if isinstance(res, str):
        pytest.fail(res)
    return res


def _group_results(group):
    rows = [r for r in ROWS if r.group == group]
    return _cached_child(group, ["rows"] + [r.name for r in rows], rows[0].env, timeout=1200)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [r.name for r in ROWS])
def test_dispatch_row(name):
    row = BY_NAME[name]
    res = _group_results(row.group)[name]
    assert not res["errors"], "\n".join(res["errors"])
    for what, caps, want, avoid in (("forward", res["fwd_kernels"], row.fwd, row.not_fwd), ("inverse", res["inv_kernels"], row.inv, row.not_inv)):
        assert sorted(caps) == sorted("%d,%d" % kv for kv in combos(row)), (what, sorted(caps))
        for combo, names in caps.items():
            k = int(combo.split(",")[0])
            for p, ks in row.expected(want):
                if k in ks:
                    assert _ran(names, p), "%s k,video=%s: %s did not run; kernels: %s" % (what, combo, p, names)
            for p in avoid:
                assert not _ran(names, p), "%s k,video=%s: %s ran, the row is there for its fall-back; kernels: %s" % (what, combo, p, names)


def _select(sort):
    return _cached_child("select_sort" if sort else "select", ["select"], {"LFM_B200_SELECT_SORT": "1" if sort else "0"}, timeout=600)


def _f32(bits):
    return struct.unpack("<f", struct.pack("<I", bits))[0]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SELECT_FRAMES))
def test_mode_selection_against_oracle(oracle, name):
    """entropies of the eight candidates (header_version 0) against oracle.select, within the tolerance of a reordered fp32
    sum; the winner is the oracle's whenever the oracle's margin exceeds that tolerance, and on exact ties (the larger
    predictor wins, as std::map overwrite does in the reference)"""
    make, T, ways = SELECT_FRAMES[name]
    f = make()
    got_all = _select(False)
    for way in ways:
        got = got_all["%s/way%d" % (name, way)]
        want_k, want = oracle.select(f, T, way)
        e = [_f32(b) for b in got["bits"]]
        assert got["selected"] == 1
        tol = [3e-4 * max(1.0, abs(w)) for w in want]
        for k in range(8):
            assert abs(e[k] - want[k]) <= tol[k], (name, way, k, e[k], want[k])
        others = [want[k] - want[want_k] for k in range(8) if k != want_k]
        if all(d == 0 or d > tol[want_k] for d in others):          # a clear margin, or exact ties only
            assert got["predictor"] == want_k, (name, way, got["predictor"], want_k, want)


@pytest.mark.gpu
def test_mode_selection_sorted_path_bit_identical():
    """LFM_B200_SELECT_SORT=1 (stable sort instead of the next-occurrence walk) builds the same integer histograms and runs the
    same entropy kernel: bit-identical entropies and the same predictor"""
    a, b = _select(False), _select(True)
    assert a.keys() == b.keys()
    for key in a:
        assert a[key] == b[key], (key, a[key], b[key])


# ------------------------------------------------------------------------------------------------ whole files
FILE_CASES = {
    # name: (stack maker, header_version, Nnum, way, ROI lb, ROI ub (x, y, z))
    "space_k5_nnum3_1024": (lambda: base_frames(Row("", 2, (5,), (2, 1024, 1024), 3)), 8 + 5, 3, 2, (5, 900, 1), (1023, 1010, 1)),
    "tiles_video_k4_nnum121": (lambda: base_frames(Row("", 0, (4,), (3, 300, 260), 121)), 0x80 | (8 + 4), 121, 0, (100, 130, 1), (250, 299, 2)),
    "tiles_video_k2_h1": (lambda: base_frames(Row("", 0, (2,), (260, 1, 200), 13)), 0x80 | (8 + 2), 13, 0, (30, 0, 127), (199, 0, 200)),
    "tiles_k2_65537_frames": (lambda: base_frames(Row("", 0, (2,), (65537, 8, 16), 3))[np.arange(65537) % PERIOD], 8 + 2, 3, 0,
                              (3, 1, 65530), (12, 6, 65536)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FILE_CASES))
def test_file_rows(oracle, tmp_path, name):
    """new shapes through the whole file path: write_stack == oracle.write byte for byte, read_stack gives the stack back,
    read_roi gives the matching crop"""
    import lfm_b200 as L
    make, hv, T, way, lb, ub = FILE_CASES[name]
    a = np.ascontiguousarray(make())
    L.set_devices(0, 1)
    fo, fg = str(tmp_path / "o.lfm"), str(tmp_path / "g.lfm")
    rc, shv = oracle.write(a, fo, hv, T, way)
    assert rc == 0 and shv == (hv & 0x80) | ((hv & 0x7F) - 8)           # the fixed predictor, not a selected one
    L.write_stack(a, fg, header_version=hv, nnum=T, way=way)
    assert open(fg, "rb").read() == open(fo, "rb").read()
    assert np.array_equal(L.read_stack(fg, way=way), a)
    r = L.read_roi(fg, lb + (0, 0), ub + (0, 0), way=way)
    assert np.array_equal(r[0, 0], a[lb[2]:ub[2] + 1, lb[1]:ub[1] + 1, lb[0]:ub[0] + 1])


if __name__ == "__main__":
    child_main(sys.argv[1:])
