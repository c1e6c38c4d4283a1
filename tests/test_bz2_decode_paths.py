"""The bzip2 decoder (csrc/bz_decode.cu: k_huff_decode -> k_imtf -> k_inv_bwt -> k_unrle / k_unrle_flat) on streams that use
what the format allows and libbz2's own writer never does, in every kernel variant the dispatcher can pick.

A stream forge (below) writes bzip2 blocks from their MTF/RLE2 symbols, in-use map, origPtr and CRC, with a chosen number of
tables (2-6), any selector sequence and surplus selectors, code lengths 1-20 (incomplete codes included) assigned canonically
as BZ2_hbAssignCodes does, lengths delta coded as libbz2 writes them or with +1 -1 detours, and the randomised bit.  The
symbols come from oracle.bz2_compress(trace=True), so the blocks are cut as libbz2 cuts them; the few blocks libbz2 never
makes (exactly 100000 * level bytes, one lap of period 2 filling a level-9 block) come from a numpy rotation sort and MTF,
checked against the oracle's trace on ordinary blocks.

A row of ROWS is a name, the data, the level and the forge options (None: the plain bz2.compress stream).  Without a GPU:
every row's stream gives the row's bytes through the system libbz2 (and the oracle's decoder where it reads the row), rows
libbz2 must reject are rejected, and each forged stream has the property its row is named for.  KLB_ROWS are .lfm files whose
blocks (raw pixels, header_version 8) are re-encoded by the forge; they read back through oracle.read.

On the GPU every row goes through bz2_decompress (k_huff_decode<*, true>, k_unrle_flat) and every KLB row through read_stack
on the host and into device memory (k_huff_decode<*, false>, k_unrle).  The switches LFM_B200_DEC_LB, LFM_B200_IBWT_NT and
LFM_B200_GROUPS are read once per process, so each group of rows runs in a fresh child process with every inherited
LFM_B200_* variable removed, at most once per test session.  One torch.profiler capture per row must list the kernel
variant the row is for, and not the one a fall-back row exists to avoid.
"""
import bz2
import heapq
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import Oracle, lf_synth

BLOCK_MAGIC = 0x314159265359
EOS_MAGIC = 0x177245385090
GSIZE = 50


# ------------------------------------------------------------------------------------------------ bits
class Bits:
    """MSB-first bit writer over numpy arrays: put() one value, put_many() arrays of values and widths"""

    def __init__(self):
        self.parts = []

    def put(self, nbits, v):
        self.put_many([v], [nbits])

    def put_many(self, values, widths):
        values = np.asarray(values, np.uint64); widths = np.asarray(widths, np.int64)
        if values.size == 0:
            return
        sh = widths[:, None] - 1 - np.arange(int(widths.max()))[None, :]
        keep = sh >= 0
        b = (values[:, None] >> np.where(keep, sh, 0).astype(np.uint64)) & np.uint64(1)
        self.parts.append(b[keep].astype(np.uint8))

    def append(self, bits):
        self.parts.append(np.asarray(bits, np.uint8))

    def bits(self):
        return np.concatenate(self.parts) if self.parts else np.zeros(0, np.uint8)


def pack(bits):
    return np.packbits(bits).tobytes()


_CRC_TAB = None


def crc32_bzip2(data):
    """bzip2's block CRC (CRC-32, MSB first), table driven"""
    global _CRC_TAB
    if _CRC_TAB is None:
        t = []
        for i in range(256):
            c = i << 24
            for _ in range(8):
                c = ((c << 1) ^ 0x04C11DB7) & 0xFFFFFFFF if c & 0x80000000 else (c << 1) & 0xFFFFFFFF
            t.append(c)
        _CRC_TAB = t
    crc, tab = 0xFFFFFFFF, _CRC_TAB
    for b in bytes(data):
        crc = ((crc << 8) & 0xFFFFFFFF) ^ tab[(crc >> 24) ^ b]
    return crc ^ 0xFFFFFFFF


# ------------------------------------------------------------------------------------------------ blocks libbz2 never cuts
def rotation_sort(t):
    """sorted rotations of the block t (prefix doubling on cyclic ranks): the last column and origPtr, as BZ2_blockSort"""
    t = np.asarray(t, np.uint8); n = len(t)
    idx = np.arange(n)
    rank = t.astype(np.int64)
    sa = np.argsort(rank, kind="stable")
    ndist, k = len(np.unique(rank)), 1
    while ndist < n:
        key2 = rank[(idx + k) % n]
        sa = np.lexsort((key2, rank))
        chg = np.concatenate([[0], np.cumsum((rank[sa][1:] != rank[sa][:-1]) | (key2[sa][1:] != key2[sa][:-1]))])
        new = np.empty(n, np.int64); new[sa] = chg
        nd = int(chg[-1]) + 1
        rank, k = new, 2 * k
        if nd == ndist:                    # classes stopped splitting: an exactly periodic block, its equal rotations stay tied
            break
        ndist = nd
    return t[(sa - 1) % n], int(np.nonzero(sa == 0)[0][0])


def mtf_rle2(last):
    """generateMTFValues (compress.c:115-235): MTF + RUNA/RUNB coding of the last column -> (mtfv with EOB, in-use byte values)"""
    last = np.asarray(last, np.uint8)
    used = np.unique(last)
    seq = np.full(256, -1, np.int64); seq[used] = np.arange(len(used))
    ll = seq[last]
    starts = np.concatenate([[0], np.nonzero(ll[1:] != ll[:-1])[0] + 1])
    lens = np.diff(np.concatenate([starts, [len(ll)]]))
    yy = list(range(len(used)))
    out = []

    def flush(z):
        z -= 1
        while True:
            out.append(1 if z & 1 else 0)
            if z < 2:
                break
            z = (z - 2) // 2

    for s, ln in zip(starts, lens):
        v = int(ll[s])
        if yy[0] == v:
            z = int(ln)
        else:
            j = yy.index(v); yy.pop(j); yy.insert(0, v)
            out.append(j + 1)
            z = int(ln) - 1
        if z:
            flush(z)
    out.append(len(used) + 1)
    return np.array(out, np.uint16), [int(u) for u in used]


def numpy_block(text):
    """one block of post-RLE1 text without runs of 4 (so the text is also the block's output): symbols, in-use, origPtr, CRC"""
    t = np.frombuffer(bytes(text), np.uint8)
    assert not np.any((t[3:] == t[2:-1]) & (t[2:-1] == t[1:-2]) & (t[1:-2] == t[:-3])), "text has a run of 4"
    last, orig = rotation_sort(t)
    mtfv, used = mtf_rle2(last)
    return dict(mtfv=mtfv, in_use=used, orig_ptr=orig, crc=crc32_bzip2(t), n=len(t))


def oracle_blocks(oracle, data, level):
    """libbz2's blocks of data at level (the oracle's trace): symbols, in-use, origPtr, CRC"""
    _, blocks = oracle.bz2_compress(data, level, trace=True)
    return [dict(mtfv=b["mtfv"].astype(np.uint16), in_use=[int(v) for v in np.unique(b["rle1"])], orig_ptr=b["orig_ptr"],
                 crc=b["crc"], n=b["nblock"]) for b in blocks]


# ------------------------------------------------------------------------------------------------ the forge
def huffman_lengths(freq, limit):
    """code lengths as BZ2_hbMakeCodeLengths builds them: Huffman over max(freq, 1), weights halved until none exceeds limit"""
    w = np.maximum(np.asarray(freq, np.int64), 1)
    while True:
        heap = [(int(x), i, (i,)) for i, x in enumerate(w)]
        heapq.heapify(heap)
        depth = np.zeros(len(w), np.int64)
        k = len(w)
        while len(heap) > 1:
            a, b = heapq.heappop(heap), heapq.heappop(heap)
            for s in a[2] + b[2]:
                depth[s] += 1
            heapq.heappush(heap, (a[0] + b[0], k, a[2] + b[2])); k += 1
        if depth.max() <= limit:
            return np.maximum(depth, 1)
        w = 1 + w // 2


def canonical_codes(lens):
    """BZ2_hbAssignCodes: codes in (length, symbol) order"""
    code = np.zeros(len(lens), np.int64)
    vec = 0
    for n in range(int(lens.min()), int(lens.max()) + 1):
        for i in np.nonzero(lens == n)[0]:
            code[i] = vec; vec += 1
        vec <<= 1
    return code


def default_tables(n_mtf):
    return 2 if n_mtf < 200 else 3 if n_mtf < 600 else 4 if n_mtf < 1200 else 5 if n_mtf < 2400 else 6


def forge_block(blk, tables=None, sel=None, nsel=None, lens=None, delta="libbz2", start=None, randomised=0, limit=17, seed=0):
    """one bzip2 block (from its magic to its last symbol) as a bit array, and what it holds.
    tables: 2..6 (default: libbz2's rule by nMTF); sel: table of every needed group (list or function of the group index);
    nsel: selectors written (>= needed: the surplus ones name random tables); lens: function (lengths[ngroups][alpha], freq,
    mtfv, sel) -> lengths, applied after the per-table Huffman limited to `limit` bits; delta: "libbz2" (runs of equal
    deltas), "zigzag" (a +1 -1 or -1 +1 detour before every third symbol), "above20" / "below1" (one record that starts at
    20 / 1 detours to 21 / 0 and back: an invalid stream whose lengths all end in range); start: per-table 5-bit start value (default:
    the first symbol's length)."""
    mtfv = np.asarray(blk["mtfv"], np.int64)
    n_mtf = len(mtfv)
    in_use = blk["in_use"]
    alpha = len(in_use) + 2
    assert int(mtfv[-1]) == alpha - 1 and mtfv.max() == alpha - 1
    ng = tables or default_tables(n_mtf)
    need = (n_mtf + GSIZE - 1) // GSIZE
    rng = np.random.default_rng(seed)
    if sel is None:
        sels = np.arange(need) % ng
    elif callable(sel):
        sels = np.array([sel(g) for g in range(need)], np.int64)
    else:
        sels = np.asarray(sel, np.int64)
    assert len(sels) == need and sels.max() < ng
    nsel = need if nsel is None else nsel
    assert need <= nsel <= 32767
    all_sel = np.concatenate([sels, rng.integers(0, ng, nsel - need)])
    grp_tab = sels[np.arange(n_mtf) // GSIZE]
    L = np.zeros((ng, alpha), np.int64)
    for t in range(ng):
        L[t] = huffman_lengths(np.bincount(mtfv[grp_tab == t], minlength=alpha), limit)
    if lens is not None:
        L = np.asarray(lens(L.copy(), np.bincount(mtfv, minlength=alpha), mtfv, sels), np.int64)
    assert L.min() >= 1 and L.max() <= 20
    for t in range(ng):
        assert np.sum(1 << (20 - L[t])) <= 1 << 20, "Kraft sum over 1"
    w = Bits()
    w.put(48, BLOCK_MAGIC); w.put(32, blk["crc"]); w.put(1, randomised); w.put(24, blk["orig_ptr"])
    used = np.zeros(256, bool); used[in_use] = True
    rows = used.reshape(16, 16)
    w.put(16, int(sum(1 << (15 - i) for i in range(16) if rows[i].any())))
    for i in range(16):
        if rows[i].any():
            w.put(16, int(sum(1 << (15 - j) for j in range(16) if rows[i, j])))
    w.put(3, ng); w.put(15, nsel)
    pos, mtfpos = list(range(ng)), []
    for s in all_sel:
        j = pos.index(int(s)); pos.pop(j); pos.insert(0, int(s)); mtfpos.append(j)
    mtfpos = np.array(mtfpos, np.int64)
    w.put_many((1 << (mtfpos + 1)) - 2, mtfpos + 1)          # j ones then a zero
    max_pairs, mixed, out_of_range = 0, False, 0
    for t in range(ng):
        curr = int(L[t, 0]) if start is None else start[t]
        w.put(5, curr)
        vals, wid = [], []
        for i in range(alpha):
            pairs = []
            if delta == "zigzag" and i % 3 == 0:
                pairs += [2, 3] if curr < 20 else [3, 2]
            if (delta, curr) in (("above20", 20), ("below1", 1)) and not out_of_range:
                pairs += [2, 3] if curr == 20 else [3, 2]
                out_of_range += 1
            target = int(L[t, i])
            pairs += [2] * max(0, target - curr) + [3] * max(0, curr - target)
            curr = target
            max_pairs = max(max_pairs, len(pairs))
            mixed = mixed or len(set(pairs)) > 1
            vals += pairs + [0]; wid += [2] * len(pairs) + [1]
        w.put_many(vals, wid)
    codes = [canonical_codes(L[t]) for t in range(ng)]
    C = np.array(codes)
    w.put_many(C[grp_tab, mtfv], L[grp_tab, mtfv])
    sym_len = L[grp_tab, mtfv]
    info = dict(n_groups=ng, n_sel=nsel, needed=need, n_mtf=n_mtf, alpha=alpha, sel_mtf_positions=sorted(set(mtfpos.tolist())),
                max_len=int(L.max()), min_len=int(L.min()), max_used_len=int(sym_len.max()), eob_len=int(sym_len[-1]),
                max_pairs=max_pairs, mixed=mixed, out_of_range=out_of_range, tables_used=sorted(set(sels.tolist())), lens=L, sym_len=sym_len,
                kraft=[int(np.sum(1 << (20 - L[t]))) for t in range(ng)], randomised=randomised)
    return w.bits(), info


def split_stream(z, nblocks):
    """the blocks of a libbz2 stream as bit arrays (magic to last symbol), found by their magics"""
    bits = np.unpackbits(np.frombuffer(z, np.uint8))
    s = bits.tobytes().replace(b"\x01", b"1").replace(b"\x00", b"0")
    bm, em = format(BLOCK_MAGIC, "048b").encode(), format(EOS_MAGIC, "048b").encode()
    starts, p = [], 32
    while len(starts) < nblocks:
        starts.append(p)
        p = s.find(bm, p + 48) if len(starts) < nblocks else s.rfind(em)
    assert s.rfind(em) > starts[-1]
    ends = starts[1:] + [s.rfind(em)]
    assert s.count(bm) == nblocks                         # no false magic: the split is exact
    return [bits[a:b] for a, b in zip(starts, ends)]


def make_stream(level, block_bits, crcs):
    w = Bits()
    for ch in b"BZh%d" % level:
        w.put(8, ch)
    comb = 0
    for b, c in zip(block_bits, crcs):
        w.append(b)
        comb = ((comb << 1) | (comb >> 31)) & 0xFFFFFFFF ^ c
    w.put(48, EOS_MAGIC); w.put(32, comb)
    return pack(w.bits())


def forge_stream(oracle, data, level, opts):
    """data at level: libbz2's block cuts, each block forged with opts (a dict for all blocks, or one entry per block: None keeps
    libbz2's own bits); opts None: bz2.compress.  Returns (stream, [info per block, None for plain blocks], blocks)"""
    blocks = oracle_blocks(oracle, data, level)
    if opts is None:
        return bz2.compress(data, level), [None] * len(blocks), blocks
    per = opts if isinstance(opts, list) else [opts] * len(blocks)
    assert len(per) == len(blocks)
    plain = split_stream(bz2.compress(data, level), len(blocks)) if any(o is None for o in per) else None
    bits, infos = [], []
    for k, (b, o) in enumerate(zip(blocks, per)):
        if o is None:
            bits.append(plain[k]); infos.append(None)
        else:
            bb, info = forge_block(b, **o); bits.append(bb); infos.append(info)
    return make_stream(level, bits, [b["crc"] for b in blocks]), infos, blocks


# ------------------------------------------------------------------------------------------------ length patterns
def max_exactly(n):
    """maximum code length exactly n: the rarest symbol the block uses gets n bits (Huffman limited to n before)"""
    def f(L, freq, mtfv, sels):
        L = np.minimum(L, n)
        used = np.nonzero(freq)[0]
        rare = used[np.argmin(freq[used])]
        L[:, rare] = n
        return L
    return f


def long_sym(pick, n=18):
    """the symbol pick(mtfv) gets n bits in every table"""
    def f(L, freq, mtfv, sels):
        L[:, pick(mtfv)] = n
        return L
    return f


def at_run_position(k):
    """a symbol that occurs at a group position p < 48 with p % 3 == k (position k of a three-symbol run) and nowhere in the
    first group at another run position, chosen among the rarest"""
    def pick(mtfv):
        p = np.arange(len(mtfv)) % GSIZE
        cand = [int(s) for s in np.unique(mtfv[:-1][(p[:-1] < 48) & (p[:-1] % 3 == k)]) if s > 1]
        freq = np.bincount(mtfv)
        return min(cand, key=lambda s: (freq[s], s))
    return pick


def in_eob_group(mtfv):
    """a symbol of the EOB group other than the one just before EOB"""
    g0 = (len(mtfv) - 1) // GSIZE * GSIZE
    last = int(mtfv[-2])
    cand = [int(s) for s in mtfv[g0:-2] if s != last and s > 1]
    freq = np.bincount(mtfv)
    return min(cand, key=lambda s: (freq[s], s))


def eob_long(L, freq, mtfv, sels):
    L[:, len(freq) - 1] = 20
    return L


def one_and_twenty(jump):
    """the most frequent symbol gets 1 bit, the others Huffman codes in the other half of the code space, the rarest used one
    20 bits; with jump, the symbol after the 1-bit one (alphabet order) also gets 20: a record of 19 +1 steps"""
    def f(L, freq, mtfv, sels):
        top = int(np.argmax(freq))
        rest = [i for i in range(len(freq)) if i != top]
        sub = huffman_lengths(freq[rest], 18) + 1
        for t in range(L.shape[0]):
            L[t, rest] = sub; L[t, top] = 1
        used = [i for i in np.nonzero(freq)[0] if i != top]
        L[:, min(used, key=lambda s: (freq[s], s))] = 20
        if jump:
            L[:, top + 1 if top + 1 < len(freq) else top - 1] = 20
        return L
    return f


# ------------------------------------------------------------------------------------------------ data
def norun(n, seed, values=None):
    """n bytes without two equal neighbours (so no RLE1 records): random over `values` (default all 256)"""
    rng = np.random.default_rng(seed)
    v = np.arange(256, dtype=np.uint8) if values is None else np.asarray(values, np.uint8)
    a = v[rng.integers(0, len(v), n)]
    for i in range(1, n):
        if a[i] == a[i - 1]:
            a[i] = v[(int(np.nonzero(v == a[i])[0][0]) + 1) % len(v)]
    return a.tobytes()


def u16(v, n):
    return np.full(n, v, "<u2").tobytes()


def skewed(n, seed):
    """uint16 Poisson noise: many distinct symbols with very unequal frequencies (long Huffman codes have rare symbols)"""
    return np.random.default_rng(seed).poisson(30, n // 2).astype("<u2").tobytes()


def eob_at(pos, seed):
    """a small-alphabet input whose stream at level 1 has EOB at group position `pos` (searched, deterministic)"""
    o = Oracle()
    rng = np.random.default_rng(seed)
    for m in range(400, 4000):
        d = rng.poisson(3, m).astype(np.uint8).tobytes()
        if (len(oracle_blocks(o, d, 1)[0]["mtfv"]) - 1) % GSIZE == pos:
            return d
    raise AssertionError("no input puts EOB at group position %d" % pos)


def text_runs(reps, seed):
    """English-like words, repeated: long equal-byte runs in the last column, hence long RUNA/RUNB sequences"""
    rng = np.random.default_rng(seed)
    words = [b"light", b"field", b"micro", b"lens", b"stack", b"frame", b"pixel", b"block"]
    return b" ".join(words[i] for i in rng.integers(0, len(words), reps)) + norun(300, seed)


# ------------------------------------------------------------------------------------------------ rows
class Row:
    def __init__(self, name, data, level, opts, check=None, reject=False, oracle_reads=True, device=False, raw=None,
                 randomised=False):
        self.name, self.data, self.level, self.opts = name, data, level, opts
        self.check = check                  # check(infos, blocks) -> truth of the row's property
        self.reject = reject                # libbz2 (and the GPU, with code 2) must reject the stream
        self.oracle_reads = oracle_reads    # the oracle's decoder reads at most 18002 selectors
        self.device = device                # also decoded from a CUDA tensor
        self.raw = raw                      # blocks libbz2 never cuts: this post-RLE1 text as ONE block (numpy_block)
        self.randomised = randomised        # the oracle's randomised-block writer


def _periodic(r):
    """the block is u repeated r times: n / (smallest cyclic period) == r"""
    def check(infos, blocks):
        return any(_block_reps(b) >= r for b in blocks)
    return check


def _block_reps(b):
    """repeats of the smallest period of a block's text, from its symbols"""
    mtfv = [int(s) for s in b["mtfv"][:-1]]
    mtf, last, run, w = list(b["in_use"]), [], 0, 1
    for s in mtfv:
        if s <= 1:
            run += (s + 1) * w; w <<= 1
            continue
        last += [mtf[0]] * run; run, w = 0, 1
        c = mtf.pop(s - 1); mtf.insert(0, c); last.append(c)
    last += [mtf[0]] * run
    L = np.array(last, np.uint8)
    P = np.argsort(L, kind="stable")
    p0 = int(P[b["orig_ptr"]]); p, c = int(P[p0]), 1
    while p != p0:
        p, c = int(P[p]), c + 1
    return len(L) // c


def _info(pred):
    return lambda infos, blocks: all(pred(i) for i in infos if i is not None) and any(i is not None for i in infos)


def _runs(mtfv):
    """(start, length) of every RUNA/RUNB sequence"""
    m = np.concatenate([[False], np.asarray(mtfv) <= 1, [False]])
    d = np.diff(m.astype(np.int8))
    a, b = np.nonzero(d == 1)[0], np.nonzero(d == -1)[0]
    return list(zip(a.tolist(), (b - a).tolist()))


def _chunk_size(b):
    nsym = len(b["mtfv"]) - 1
    return (nsym + 127) // 128


def _long_at_run_pos(k):
    def check(infos, blocks):
        i, b = infos[0], blocks[0]
        p = np.arange(len(b["mtfv"])) % GSIZE
        return bool(np.any((i["sym_len"] > 10) & (p < 48) & (p % 3 == k)))
    return check


def _long_in_eob_group(infos, blocks):
    i, b = infos[0], blocks[0]
    g0 = (len(b["mtfv"]) - 1) // GSIZE * GSIZE
    return bool(np.any(i["sym_len"][g0:-2] > 10)) and i["sym_len"][-2] <= 10


_SKEW = lambda: skewed(60000, 5)
_R = "libbz2"
ROWS = [
    # ---- exactly periodic blocks (the plain stream)
    *[Row("const%d_%dpx" % (v, n), (lambda v=v, n=n: u16(v, n)), 9, None, check=_periodic(n), device=(n == 73728))
      for v in (100, 300) for n in (9216, 18432, 73728, 100000)],
    Row("const300_level9_block_900000", lambda: u16(300, 450000), 9, {}, raw=True, check=_periodic(450000)),
    Row("abc_x13000", lambda: b"abc" * 13000, 1, None, check=_periodic(13000)),
    Row("zero_runs_block", lambda: bytes(255 * 19997), 1, None, check=_periodic(19997)),
    Row("period1500_r3", lambda: norun(1500, 3) * 3, 1, None, check=_periodic(3)),
    Row("randomised_periodic", lambda: u16(300, 9216), 1, None, randomised=True),
    # ---- long codes
    *[Row("max_len_%d" % n, _SKEW, 1, dict(lens=max_exactly(n), limit=n), check=_info(lambda i, n=n: i["max_len"] == n and i["max_used_len"] == n))
      for n in (9, 10, 11, 17, 18, 20)],
    Row("eob_20_bits", _SKEW, 1, dict(lens=eob_long), check=_info(lambda i: i["eob_len"] == 20)),
    *[Row("long_code_run_pos%d" % k, _SKEW, 1, dict(lens=long_sym(at_run_position(k))), check=_long_at_run_pos(k)) for k in range(3)],
    Row("long_code_before_eob", _SKEW, 1, dict(lens=long_sym(lambda m: int(m[-2]), 20)), check=_info(lambda i: i["sym_len"][-2] == 20)),
    Row("long_code_in_eob_group", _SKEW, 1, dict(lens=long_sym(in_eob_group, 19)), check=_long_in_eob_group),
    # ---- code-length records
    Row("mixed_deltas", _SKEW, 1, dict(delta="zigzag"), check=_info(lambda i: i["mixed"])),
    Row("lengths_1_and_20", _SKEW, 1, dict(lens=one_and_twenty(False)), check=_info(lambda i: i["min_len"] == 1 and i["max_len"] == 20)),
    Row("jump_1_to_20", _SKEW, 1, dict(lens=one_and_twenty(True)), check=_info(lambda i: i["max_pairs"] >= 19)),
    # a detour out of 1..20 inside one record: libbz2 checks every step; the final lengths are valid, so only a per-step check
    # (the bit-by-bit loop that mixed deltas take) rejects it
    Row("detour_above_20_rejected", _SKEW, 1, dict(lens=one_and_twenty(False), delta="above20"), reject=True,
        check=_info(lambda i: i["out_of_range"] == 1)),
    Row("detour_below_1_rejected", _SKEW, 1, dict(lens=one_and_twenty(False), delta="below1"), reject=True,
        check=_info(lambda i: i["out_of_range"] == 1)),
    Row("start_far_from_first_length", _SKEW, 1, dict(start=[20, 1, 20, 1, 20, 1]), check=_info(lambda i: i["max_pairs"] >= 16)),
    Row("alpha258_mixed", lambda: norun(40000, 7), 1, dict(delta="zigzag", lens=max_exactly(20)),
        check=_info(lambda i: i["alpha"] == 258 and i["mixed"])),
    Row("alpha258_jumps", lambda: norun(40000, 8), 1, dict(lens=one_and_twenty(True)),
        check=_info(lambda i: i["alpha"] == 258 and i["max_pairs"] >= 19)),
    # ---- tables and selectors
    Row("tables6_nmtf_lt_200", lambda: norun(150, 9, range(40)), 1, dict(tables=6), check=_info(lambda i: i["n_groups"] == 6 and i["n_mtf"] < 200)),
    Row("tables2_nmtf_gt_2400", _SKEW, 1, dict(tables=2), check=_info(lambda i: i["n_groups"] == 2 and i["n_mtf"] > 2400)),
    Row("unused_table", _SKEW, 1, dict(tables=4, sel=lambda g: (0, 1, 3)[g % 3]), check=_info(lambda i: i["tables_used"] == [0, 1, 3])),
    Row("every_selector_mtf_position", _SKEW, 1, dict(tables=6, sel=lambda g: (g * g + 3 * g) % 7 % 6),
        check=_info(lambda i: i["sel_mtf_positions"] == [0, 1, 2, 3, 4, 5])),
    Row("surplus_selectors_plus1", _SKEW, 1, dict(nsel=-1), check=_info(lambda i: i["n_sel"] == i["needed"] + 1)),
    *[Row("surplus_selectors_%d" % n, _SKEW, 1, dict(nsel=n, tables=6), check=_info(lambda i, n=n: i["n_sel"] == n),
          oracle_reads=n <= 18002, device=(n == 32767)) for n in (18002, 20001, 32767)],
    # ---- alphabet
    Row("alphabet_one_value", lambda: bytes([251]) * (255 * 40), 1, dict(tables=3), check=_info(lambda i: i["alpha"] == 3)),
    Row("alphabet_one_byte_block", lambda: b"x", 1, dict(tables=6), check=_info(lambda i: i["alpha"] == 3)),
    Row("alphabet_256", lambda: norun(20000, 11), 1, dict(delta="zigzag"), check=_info(lambda i: i["alpha"] == 258)),
    Row("alphabet_0_and_255", lambda: norun(20000, 12, (0, 255)), 1, {}, check=_info(lambda i: i["alpha"] == 4)),
    # ---- EOB position in its group
    *[Row("eob_group_pos%d" % p, (lambda p=p: eob_at(p, 20 + p)), 1, {}, check=_info(lambda i, p=p: (i["n_mtf"] - 1) % GSIZE == p))
      for p in (0, 31, 32, 49)],
    # ---- RUNA / RUNB sequences
    # (the first symbol is a run only in a block whose smallest rotation follows its smallest byte: a constant block)
    Row("run_at_first_symbol", lambda: bytes([251]) * (255 * 333), 1, dict(tables=5, delta="zigzag"), check=lambda infos, blocks: int(blocks[0]["mtfv"][0]) <= 1),
    Row("run_longer_than_imtf_chunk", lambda: b"ab" * 3000 + norun(40, 4), 1, {},
        check=lambda infos, blocks: max(l for _, l in _runs(blocks[0]["mtfv"][:-1])) > _chunk_size(blocks[0])),
    Row("runs_straddle_imtf_chunks", lambda: text_runs(12000, 5), 1, {},
        check=lambda infos, blocks: sum(1 for a, l in _runs(blocks[0]["mtfv"][:-1]) for t in range(1, 128)
                                        if a < t * _chunk_size(blocks[0]) < a + l) >= 5),
    # ---- block size and origPtr
    Row("block_100000_level1", lambda: norun(100000, 13), 1, {}, raw=True, check=lambda infos, blocks: blocks[0]["n"] == 100000),
    Row("block_100001_level1", lambda: norun(100001, 14), 1, {}, raw=True, reject=True, check=lambda infos, blocks: blocks[0]["n"] == 100001),
    Row("orig_ptr_0", lambda: b"\x00" + norun(5000, 15, range(1, 256)), 1, {}, check=lambda infos, blocks: blocks[0]["orig_ptr"] == 0),
    Row("orig_ptr_last", lambda: b"\xff" + norun(5000, 16, range(255)), 1, {},
        check=lambda infos, blocks: blocks[0]["orig_ptr"] == blocks[0]["n"] - 1),
    Row("one_byte_block", lambda: b"q", 9, None),
    # ---- streams
    Row("multi_block_forged_and_plain", lambda: skewed(420000, 17), 1,
        [None, dict(delta="zigzag", lens=max_exactly(20)), None, dict(tables=6, nsel=-1), dict(lens=eob_long)],
        check=lambda infos, blocks: len(blocks) == 5, device=True),
]
BY_NAME = {r.name: r for r in ROWS}
assert len(BY_NAME) == len(ROWS)

CONCAT = ["const300_18432px", "max_len_20", "surplus_selectors_18002", "one_byte_block", "alphabet_0_and_255", "abc_x13000"]


_built = {}


def build_row(oracle, row):
    """(stream, expected bytes, infos, blocks) of a row, built once per process"""
    if row.name in _built:
        return _built[row.name]
    data = row.data()
    if row.name == "concatenated_levels":
        parts = [build_row(oracle, BY_NAME[n]) for n in CONCAT]
        res = (b"".join(p[0] for p in parts), b"".join(p[1] for p in parts), [], [])
    elif row.randomised:
        oracle.set_randomised(True)
        try:
            z = oracle.bz2_compress(data, row.level)
        finally:
            oracle.set_randomised(False)
        res = (z, data, [], [])
    elif row.raw:
        blk = numpy_block(data)
        bits, info = forge_block(blk, **row.opts)
        res = (make_stream(row.level, [bits], [blk["crc"]]), data, [info], [blk])
    else:
        opts = row.opts
        if isinstance(opts, dict) and opts.get("nsel") == -1 or isinstance(opts, list):
            blocks = oracle_blocks(oracle, data, row.level)
            fix = lambda o, b: o if o is None or o.get("nsel") != -1 else dict(o, nsel=(len(b["mtfv"]) + GSIZE - 1) // GSIZE + 1)
            opts = [fix(o, b) for o, b in zip(opts if isinstance(opts, list) else [opts] * len(blocks), blocks)]
        z, infos, blocks = forge_stream(oracle, data, row.level, opts)
        res = (z, data, infos, blocks)
    _built[row.name] = res
    return res


ROWS.append(Row("concatenated_levels", lambda: b"", 0, None, oracle_reads=False, device=True))
BY_NAME["concatenated_levels"] = ROWS[-1]


# ------------------------------------------------------------------------------------------------ KLB rows
class KlbRow:
    def __init__(self, name, img, bs, opts, small=False, many=False):
        self.name, self.img, self.bs, self.opts = name, img, bs, opts   # bs: (x, y, z) block size
        self.small = small                  # slots of <= 48 KB: k_inv_bwt<256> unless LFM_B200_IBWT_NT=1024
        self.many = many                    # more blocks than 10-bit tables keep resident: k_huff_decode<9, false>


def _pairs_img(shape, seed):
    """pixels v * 257 in equal pairs along x: every 4 bytes equal, so RLE1 writes 5 bytes for 4 (two bzip2 blocks per 409600)"""
    rng = np.random.default_rng(seed)
    Z, Y, X = shape
    v = rng.integers(0, 255, (Z, Y, X // 2))
    v[..., 1:] += (v[..., 1:] == v[..., :-1])
    return (np.repeat(v, 2, axis=2) * 257).astype(np.uint16)


_L20 = dict(lens=max_exactly(20), delta="zigzag")
KLB_ROWS = [
    KlbRow("klb_const300_96x96x8", lambda: np.full((16, 96, 96), 300, np.uint16), (96, 96, 8), None),
    KlbRow("klb_const100_96x96x2", lambda: np.full((4, 96, 96), 100, np.uint16), (96, 96, 2), None, small=True),
    KlbRow("klb_synth_96x96x2_long_mixed", lambda: lf_synth((6, 192, 96), 13, seed=3), (96, 96, 2), _L20, small=True),
    KlbRow("klb_synth_96x96x2_tables6_surplus", lambda: lf_synth((4, 96, 192), 13, seed=4), (96, 96, 2), dict(tables=6, nsel=18002), small=True),
    KlbRow("klb_synth_96x96x8_long_mixed", lambda: lf_synth((16, 96, 96), 13, seed=5), (96, 96, 8), _L20),
    KlbRow("klb_synth_96x96x8_surplus", lambda: lf_synth((8, 96, 96), 13, seed=6), (96, 96, 8), dict(nsel=18002, lens=eob_long)),
    KlbRow("klb_pairs_160x160x8_two_bz_blocks", lambda: _pairs_img((8, 160, 160), 7), (160, 160, 8),
           [None, dict(lens=one_and_twenty(True), tables=6)]),
    KlbRow("klb_2400_blocks_16x16x1", lambda: lf_synth((24, 160, 160), 13, seed=8), (16, 16, 1), dict(lens=max_exactly(18)),
           small=True, many=True),
]
KLB_BY_NAME = {r.name: r for r in KLB_ROWS}


def klb_blocks(img, bs):
    """(z, y, x) boxes of the KLB blocks in file order (x fastest)"""
    Z, Y, X = img.shape
    bx, by, bz = bs
    return [(z, y, x) for z in range(0, Z, bz) for y in range(0, Y, by) for x in range(0, X, bx)]


def build_klb(oracle, row, path):
    """the row's .lfm file (stored header version 0: what header_version 8 writes, no predictor) and its image; the forged
    blocks' infos"""
    from importlib import import_module
    D = import_module("lightfieldmicroscopy_pc-bzip2_b200.distributed")
    img = row.img()
    Z, Y, X = img.shape
    bx, by, bz = row.bs
    level = min(9, -(-bx * by * bz * 2 // 100000))
    streams, infos = [], []
    for z, y, x in klb_blocks(img, row.bs):
        raw = np.ascontiguousarray(img[z:z + bz, y:y + by, x:x + bx]).tobytes()
        opts = row.opts
        if isinstance(opts, list):
            nb = len(oracle_blocks(oracle, raw, level))
            opts = opts[:nb] if nb == len(opts) else opts[-1]
        s, inf, _ = forge_stream(oracle, raw, level, opts)
        streams.append(s); infos += inf
    off = np.cumsum([len(s) for s in streams])
    with open(path, "wb") as f:
        f.write(D.pack_header(0, 13, (X, Y, Z, 1, 1), (bx, by, bz, 1, 1), off))
        for s in streams:
            f.write(s)
    return img, infos


# ------------------------------------------------------------------------------------------------ no GPU needed
@pytest.mark.parametrize("name", [r.name for r in ROWS])
def test_row_stream_read_by_libbz2(oracle, name):
    """the system libbz2 gives the row's bytes (or rejects a stream it must reject), and so does the oracle's decoder where it
    reads the row"""
    row = BY_NAME[name]
    z, want, infos, blocks = build_row(oracle, row)
    if row.reject:
        with pytest.raises(OSError):
            bz2.decompress(z)
        assert oracle.bz2_decompress(z, len(want) + 1000)[0] != 0
        return
    assert bz2.decompress(z) == want
    if row.oracle_reads:
        rc, got = oracle.bz2_decompress(z, len(want) + 1000)
        assert rc == 0 and got == want


@pytest.mark.parametrize("name", [r.name for r in ROWS if r.check is not None])
def test_row_has_its_property(oracle, name):
    """each forged stream has what its row is named for (maximum code length, selector count, EOB position, ...)"""
    row = BY_NAME[name]
    _, _, infos, blocks = build_row(oracle, row)
    assert row.check(infos, blocks), name


def test_numpy_block_matches_oracle(oracle):
    """the rotation sort and MTF of the test, against libbz2's blocks as the oracle traces them"""
    for data, level in ((skewed(30000, 1), 1), (norun(5000, 2), 1), (b"ab" * 700 + b"c", 1), (text_runs(3000, 3), 2)):
        _, blocks = oracle.bz2_compress(data, level, trace=True)
        for b in blocks:
            last, orig = rotation_sort(b["rle1"])
            assert np.array_equal(last, b["bwt"]) and orig == b["orig_ptr"]
            mtfv, used = mtf_rle2(b["bwt"])
            assert np.array_equal(mtfv, b["mtfv"])
            assert crc32_bzip2(data) == b["crc"] or len(blocks) > 1


def test_forge_with_libbz2_table_count_is_readable(oracle):
    """the forge with libbz2's table count gives a stream libbz2 reads (the baseline every forged row departs from)"""
    data = skewed(150000, 9)
    z, infos, blocks = forge_stream(oracle, data, 1, {})
    assert len(blocks) == 2 and bz2.decompress(z) == data


def test_klb_builder_matches_oracle_write(oracle, tmp_path):
    """a KLB file built here with libbz2's plain streams equals oracle.write(header_version 8) byte for byte"""
    row = KlbRow("", lambda: lf_synth((5, 100, 110), 13, seed=1), (96, 96, 2), None)
    img, _ = build_klb(oracle, row, str(tmp_path / "a.lfm"))
    rc, shv = oracle.write(img, str(tmp_path / "b.lfm"), 8, 13, 0, block_size=(96, 96, 2, 1, 1))
    assert rc == 0 and shv == 0
    assert open(tmp_path / "a.lfm", "rb").read() == open(tmp_path / "b.lfm", "rb").read()


@pytest.mark.parametrize("name", [r.name for r in KLB_ROWS])
def test_klb_row_read_by_oracle(oracle, tmp_path, name):
    row = KLB_BY_NAME[name]
    path = str(tmp_path / "r.lfm")
    img, infos = build_klb(oracle, row, path)
    rc, got = oracle.read(path, img.shape, 0)
    assert rc == 0 and np.array_equal(got, img)
    if row.opts is not None:
        assert any(i is not None for i in infos)
    if name.startswith("klb_pairs_160"):
        assert len(infos) == 2 * len(klb_blocks(img, row.bs)) and infos[0] is None and infos[1]["max_len"] == 20


# ------------------------------------------------------------------------------------------------ GPU rows (child side)
GROUPS = {
    "default": {},
    "dec_lb9": {"LFM_B200_DEC_LB": "9"},
    "dec_lb10": {"LFM_B200_DEC_LB": "10"},
    "ibwt_nt1024": {"LFM_B200_IBWT_NT": "1024"},
    "groups4": {"LFM_B200_GROUPS": "4"},
}
STANDALONE_GROUPS = ("default", "dec_lb9", "dec_lb10", "ibwt_nt1024")


def expected_kernels(group, row):
    """(kernels the row's capture must list, kernels it must not list)"""
    env = GROUPS[group]
    forced = env.get("LFM_B200_DEC_LB")
    if isinstance(row, Row):
        lb = 9 if forced == "9" else 10
        must = ["k_huff_decode<%d, true>" % lb]
        if not row.reject:
            must += ["k_inv_bwt<1024>", "k_unrle_flat"]
        return must, ["k_huff_decode<%d, true>" % (19 - lb), "k_huff_decode<10, false>", "k_huff_decode<9, false>"]
    # LFM_B200_GROUPS=4 splits the 2400 blocks into launches of 600, which 10-bit tables keep resident
    lb = 9 if forced == "9" or (forced != "10" and row.many and group != "groups4") else 10
    nt = 256 if row.small and env.get("LFM_B200_IBWT_NT") != "1024" else 1024
    return (["k_huff_decode<%d, false>" % lb, "k_inv_bwt<%d>" % nt, "k_unrle<", "k_imtf"],
            ["k_huff_decode<%d, false>" % (19 - lb), "k_inv_bwt<%d>" % (1280 - nt), "true>"])


def _kernels(prof):
    return sorted({e.key for e in prof.key_averages() if "lfm::" in e.key})


def run_rows(L, cache, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    res = {}
    for name in names:
        errors, kern = [], []
        try:
            if name in BY_NAME:
                row = BY_NAME[name]
                z = open(os.path.join(cache, name + ".bz2"), "rb").read()
                want = open(os.path.join(cache, name + ".out"), "rb").read()
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    try:
                        got, code = L.bz2_decompress(z), 0
                    except L.LfmError as e:
                        got, code = None, e.code
                    torch.cuda.synchronize()
                kern = _kernels(prof)
                if row.reject:
                    if code != 2:
                        errors.append("expected code 2, got %d" % code)
                elif code:
                    errors.append("bz2_decompress: code %d (%s)" % (code, L.lib.lfmLastError().decode()))
                elif got != want:
                    errors.append("bytes differ (len %d vs %d), first at %s" % (len(got), len(want), _first(got, want)))
                if row.device and not row.reject:
                    t = torch.frombuffer(bytearray(z), dtype=torch.uint8).cuda()
                    d = bytes(L.bz2_decompress(t).cpu().numpy())
                    if d != want:
                        errors.append("device: bytes differ, first at %s" % _first(d, want))
            elif name == "write_stack_const300_hv8":
                a = np.full((16, 96, 96), 300, np.uint16)
                fn = os.path.join(cache, "ws.lfm")
                L.write_stack(a, fn, header_version=8, nnum=13, block_size=(96, 96, 8, 1, 1), way=0)
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    back = L.read_stack(fn, way=0)
                    torch.cuda.synchronize()
                kern = _kernels(prof)
                if not np.array_equal(back, a):
                    errors.append("read_stack differs from the stack written")
            else:
                fn = os.path.join(cache, name + ".lfm")
                img = np.load(os.path.join(cache, name + ".npy"))
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    back = L.read_stack(fn, way=0)
                    torch.cuda.synchronize()
                kern = _kernels(prof)
                if not np.array_equal(back, img):
                    errors.append("read_stack (host) differs, first at %s" % (np.argwhere(back != img)[:1].tolist(),))
                dev = L.read_stack(fn, way=0, device="cuda")
                if not np.array_equal(dev.cpu().numpy(), img):
                    errors.append("read_stack (device) differs")
        except Exception as e:                                           # report, and go on with the next row
            errors.append("%s: %s" % (type(e).__name__, e))
        res[name] = dict(errors=errors, kernels=kern)
    return res


def _first(a, b):
    n = min(len(a), len(b))
    x = np.frombuffer(a[:n], np.uint8) != np.frombuffer(b[:n], np.uint8)
    return int(np.argmax(x)) if x.any() else n


def child_main(argv):
    """python test_bz2_decode_paths.py CACHE NAME...: decode the rows in this (fresh) process, print one RESULT line of JSON"""
    import lfm_b200 as L
    L.set_devices(0, 1)
    print("RESULT " + json.dumps(run_rows(L, argv[0], argv[1:])), flush=True)


# ------------------------------------------------------------------------------------------------ GPU rows (pytest side)
_results = {}        # group -> the child's result, or the text of its failure: each child runs at most once per session


def _child(args, env_extra, timeout):
    env = {k: v for k, v in os.environ.items() if not k.startswith("LFM_B200_")}
    env.update(env_extra)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__)] + list(args)
    try:
        p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return "child did not finish in %d s" % timeout
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("RESULT ")]
    if p.returncode != 0 or not lines:
        return "child failed (exit %d):\n%s\n%s" % (p.returncode, p.stdout[-3000:], p.stderr[-3000:])
    return json.loads(lines[-1][len("RESULT "):])


def _names(group):
    klb = [r.name for r in KLB_ROWS] + ["write_stack_const300_hv8"]
    return klb if group == "groups4" else [r.name for r in ROWS] + klb


@pytest.fixture(scope="session")
def row_cache(tmp_path_factory):
    """every row's stream and bytes, every KLB row's file and image, written once for all children"""
    d = tmp_path_factory.mktemp("bz2_paths")
    oracle = Oracle()
    for r in ROWS:
        z, want, _, _ = build_row(oracle, r)
        open(d / (r.name + ".bz2"), "wb").write(z)
        open(d / (r.name + ".out"), "wb").write(want)
    for r in KLB_ROWS:
        img, _ = build_klb(oracle, r, str(d / (r.name + ".lfm")))
        np.save(d / (r.name + ".npy"), img)
    return str(d)


def _group_results(row_cache, group):
    if group not in _results:
        _results[group] = _child([row_cache] + _names(group), GROUPS[group], timeout=1200)
    res = _results[group]
    if isinstance(res, str):
        pytest.fail(res)
    return res


GPU_CASES = [(g, n) for g in GROUPS for n in _names(g)]


@pytest.mark.gpu
@pytest.mark.parametrize("group,name", GPU_CASES, ids=["%s-%s" % c for c in GPU_CASES])
def test_gpu_row(row_cache, group, name):
    res = _group_results(row_cache, group)[name]
    assert not res["errors"], "\n".join(res["errors"])
    if name == "write_stack_const300_hv8":
        return
    must, avoid = expected_kernels(group, BY_NAME.get(name) or KLB_BY_NAME[name])
    for p in must:
        assert any(p in k for k in res["kernels"]), "%s did not run; kernels: %s" % (p, res["kernels"])
    for p in avoid:
        assert not any(p in k for k in res["kernels"]), "%s ran; kernels: %s" % (p, res["kernels"])


if __name__ == "__main__":
    child_main(sys.argv[1:])
