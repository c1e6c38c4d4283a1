#!/usr/bin/env python3
"""record_bench.py -- a camera-style recording through StackWriter against the one-shot writeLFMstackEx of the same frames.

  python tools/record_bench.py [--frames 256] [--size 2048] [--ring 16] [--out DIR]

Frames: LF-synth (lf_synth_int, Nnum 15) of size x size uint16, a ring of `ring` distinct frames repeated, predictor way 2 (space),
headerVersion 0 (mode selection on frame 0), 96x96x1 KLB blocks.  Three files go to DIR (default /dev/shm):
  rec_host  one frame per lfmStackWriterAppend from a PAGEABLE numpy ring
  rec_dev   one frame per lfmStackWriterAppendDevice from a CUDA-tensor ring
  oneshot   writeLFMstackEx of the whole stack (pageable host memory)
All three must be byte-identical.  Reported per run: wall time open -> close (or of the writeLFMstackEx call), sustained GB/s of raw
uint16 and frames/s, p50 / p99 latency of one append, and the device memory the writer held (free memory before Open minus the
least free memory seen while recording; on the first recording of the process, so that it also counts the engine workspace the
batches use, which later calls reuse).  The card name and power limit are printed beside the numbers."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


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


def md5(fn):
    h = hashlib.md5()
    with open(fn, "rb") as f:
        for chunk in iter(lambda: f.read(1 << 24), b""):
            h.update(chunk)
    return h.hexdigest()


def record(L, fn, ring, n, H, W):
    import torch
    free0 = torch.cuda.mem_get_info()[0]
    lat = []
    least = free0
    t0 = time.perf_counter()
    w = L.StackWriter(fn, (n, H, W), header_version=0, nnum=15, block_size=(96, 96, 1, 1, 1), way=2)
    for f in range(n):
        a = time.perf_counter()
        w.append(ring[f % len(ring)])
        lat.append(time.perf_counter() - a)
        if f % 8 == 7:
            least = min(least, torch.cuda.mem_get_info()[0])
    kept = w.close()
    t = time.perf_counter() - t0
    assert kept == n
    lat = np.array(lat) * 1e3
    return dict(seconds=t, gbs=n * H * W * 2 / t / 1e9, fps=n / t, append_ms_p50=float(np.percentile(lat, 50)),
                append_ms_p99=float(np.percentile(lat, 99)), append_ms_max=float(lat.max()), device_mb_held=(free0 - least) / 2**20)



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--ring", type=int, default=16)
    ap.add_argument("--out", default="/dev/shm")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "record_bench needs a CUDA device"
    import lfm_b200 as L
    from conftest import lf_synth_int
    L.set_devices(0, 1)
    n, H, W = args.frames, args.size, args.size
    dring = lf_synth_int((args.ring, H, W), 15, seed=5, device="cuda")
    hring = dring.cpu().numpy().view(np.uint16)                     # pageable
    stack = np.ascontiguousarray(np.concatenate([hring] * ((n + args.ring - 1) // args.ring))[:n])
    files = {k: os.path.join(args.out, "lfm_record_bench_%s_%d.lfm" % (k, os.getpid())) for k in ("rec_host", "rec_dev", "oneshot")}
    try:
        # warm-up: module loads, engine workspace, the writers' staging memory
        warm = record(L, files["rec_host"], hring, min(n, 2 * args.ring), H, W)
        L.write_stack(stack[:min(n, 2 * args.ring)], files["oneshot"], header_version=0, nnum=15, block_size=(96, 96, 1, 1, 1), way=2)
        res = {"card": None, "power_limit": None, "device_mb_held": warm["device_mb_held"]}
        res["rec_host"] = record(L, files["rec_host"], hring, n, H, W)
        res["rec_dev"] = record(L, files["rec_dev"], dring, n, H, W)
        for k in ("rec_host", "rec_dev"):
            del res[k]["device_mb_held"]                             # the first recording's buffers are reused: nothing new
        t0 = time.perf_counter()
        L.write_stack(stack, files["oneshot"], header_version=0, nnum=15, block_size=(96, 96, 1, 1, 1), way=2)
        t = time.perf_counter() - t0
        res["oneshot"] = dict(seconds=t, gbs=n * H * W * 2 / t / 1e9, fps=n / t)
        sums = {k: md5(v) for k, v in files.items()}
        res["byte_identical"] = len(set(sums.values())) == 1
        res["file_bytes"] = os.path.getsize(files["oneshot"])
        res["card"], res["power_limit"] = card()
        res["workload"] = "%d frames %dx%d LF-synth, Nnum 15, way 2, auto mode, 96x96x1 blocks, one frame per append" % (n, H, W)
        print(json.dumps(res))
        if not res["byte_identical"]:
            sys.exit("recorded files differ from writeLFMstackEx: %s" % sums)
    finally:
        for v in files.values():
            if os.path.exists(v):
                os.remove(v)


if __name__ == "__main__":
    main()
