#!/usr/bin/env python3
"""playback_bench.py -- playing a recording back frame by frame through StackReader, against read_roi per frame and read_stack.

  python tools/playback_bench.py [--frames 256] [--size 2048] [--ring 16] [--reps 3] [--parent-lib PATH] [--out DIR]

A recording of `frames` LF-synth frames (lf_synth_int, Nnum 15, a ring of `ring` distinct frames) of size x size uint16 is written
with StackWriter to DIR (default /dev/shm): predictor way 2 (space), headerVersion 0 (mode selection on frame 0), 96x96x1 blocks.
Before anything is timed, every path below must return the same pixels.  Paths, each timed `reps` times:
  roi_per_frame       one read_roi (host) per time point: what playing a recording back cost before StackReader
  reader_numpy        StackReader, one frame per read, into numpy
  reader_cuda         StackReader, one frame per read, into a CUDA tensor
  read_stack          read_stack of the whole file into numpy (the full read, served by the reader)
  read_stack_parent   with --parent-lib: readKLBstackInPlace of the library built from the parent commit, in child processes that
                      alternate with children running the current library (read_stack_child), so that both see the same host
Reported: GB/s of raw uint16 pixels delivered, and p50 / p99 latency of one read for the per-frame paths.  The card name and power
limit are printed beside the numbers."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

_CHILD = """
import ctypes as C, sys, time
import numpy as np
lib = C.CDLL(sys.argv[1]); fn = sys.argv[2].encode(); n, H, W, reps = map(int, sys.argv[3:7])
lib.readKLBstackInPlace.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(C.c_int), C.c_int]
out = np.empty((n, H, W), np.uint16); dt = C.c_int()
assert lib.readKLBstackInPlace(fn, out.ctypes.data, C.byref(dt), -1) == 0            # warm-up
ts = []
for _ in range(reps):
    t0 = time.perf_counter(); assert lib.readKLBstackInPlace(fn, out.ctypes.data, C.byref(dt), -1) == 0; ts.append(time.perf_counter() - t0)
print(min(ts), float(np.median(ts)), int(out[::7, ::97, ::89].astype(np.uint64).sum()))
"""


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


def per_frame(read, n):
    lat = []
    t0 = time.perf_counter()
    for f in range(n):
        a = time.perf_counter()
        read(f)
        lat.append(time.perf_counter() - a)
    return time.perf_counter() - t0, lat


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--ring", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default="/dev/shm" if os.access("/dev/shm", os.W_OK) else "/tmp")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import lfm_b200 as L
    from conftest import lf_synth_int
    if not torch.cuda.is_available():
        sys.exit("playback_bench needs a CUDA device")
    L.set_devices(0, 1)
    n, H, W = args.frames, args.size, args.size
    ring = lf_synth_int((args.ring, H, W), 15, seed=3, device="cuda").cpu().numpy().view(np.uint16)
    fn = os.path.join(args.out, "lfm_playback_%d.lfm" % os.getpid())
    res = {}
    try:
        with L.StackWriter(fn, (n, H, W), header_version=0, nnum=15, block_size=(96, 96, 1, 1, 1), way=2) as w:
            for f in range(n):
                w.append(ring[f % args.ring])
        gb = n * H * W * 2 / 1e9
        # the same pixels on every path first
        whole = L.read_stack(fn, way=2)
        assert all(np.array_equal(whole[f], ring[f % args.ring]) for f in range(n))
        for f in (0, 1, n // 2, n - 1):
            assert np.array_equal(L.read_roi(fn, (0, 0, f, 0, 0), (W - 1, H - 1, f, 0, 0), way=2)[0, 0], whole[f:f + 1])
        with L.StackReader(fn, way=2) as r:
            for f in range(n):
                assert np.array_equal(r.read(1)[0], whole[f])
        with L.StackReader(fn, way=2, device="cuda") as r:
            for f in range(n):
                assert np.array_equal(r.read(1)[0].cpu().numpy(), whole[f])

        def report(name, secs, lat=None):
            d = dict(GBps=round(gb / secs, 2), seconds=round(secs, 3))
            if lat:
                d["p50_ms"] = round(1e3 * float(np.percentile(lat, 50)), 2)
                d["p99_ms"] = round(1e3 * float(np.percentile(lat, 99)), 2)
            res.setdefault(name, []).append(d)
            print(name, d, flush=True)

        for _ in range(args.reps):
            s, lat = per_frame(lambda f: L.read_roi(fn, (0, 0, f, 0, 0), (W - 1, H - 1, f, 0, 0), way=2), n)
            report("roi_per_frame", s, lat)
            with L.StackReader(fn, way=2) as r:
                s, lat = per_frame(lambda f: r.read(1), n)
            report("reader_numpy", s, lat)
            out = torch.empty((1, H, W), dtype=torch.uint16, device="cuda")
            with L.StackReader(fn, way=2) as r:
                s, lat = per_frame(lambda f: r.read(1, out=out), n)
            report("reader_cuda", s, lat)
            t0 = time.perf_counter()
            L.read_stack(fn, way=2)
            report("read_stack", time.perf_counter() - t0)
        if args.parent_lib:
            env = dict(os.environ, LFM_PREDICTOR_WAY="2")
            for _ in range(args.reps):
                for name, lib in (("read_stack_child", L.LIB_PATH), ("read_stack_parent", args.parent_lib)):
                    o = subprocess.run([sys.executable, "-c", _CHILD, lib, fn, str(n), str(H), str(W), "3"], env=env,
                                       capture_output=True, text=True, timeout=1200)
                    assert o.returncode == 0, o.stderr[-2000:]
                    best, med, check = o.stdout.split()
                    res.setdefault(name + "_check", set()).add(check)
                    report(name, float(best))
            for name in ("read_stack_child", "read_stack_parent"):
                res[name + "_check"] = sorted(res[name + "_check"])
            assert res["read_stack_child_check"] == res["read_stack_parent_check"], "the parent library decodes other pixels"
        name, power = card()
        res["card"] = name
        res["power_limit"] = power
        res["shape"] = [n, H, W]
        print("card: %s, power limit %s" % (name, power))
        if args.json:
            json.dump(res, open(args.json, "w"), indent=1)
    finally:
        if os.path.exists(fn):
            os.remove(fn)


if __name__ == "__main__":
    main()
