#!/usr/bin/env python3
"""Throughput of the standalone bzip2 streams (lfmBz2Compress[Device], lfmBz2Decompress[Device]) against single-core Python bz2.

Seeded inputs of --mb MiB: LF-synth frames as bytes (the integer LF-synth pattern of tests/conftest.py) and uniform random bytes.
For every input and level the GPU stream is first checked byte for byte against bz2.compress (whose time is the single-core
figure), then timed device-resident (device bytes -> device stream) and host to host (bytes -> bytes); the same for decompression of
that stream (checked against the input first).  Rates are GB/s of
uncompressed input (1e9 bytes).  Writes one JSON file with the GPU name and power limit beside the numbers; prints it too.

    python tools/bz2_bench.py --mb 256 --levels 1 9 --reps 3 --out bz2_bench.json
"""
import argparse
import bz2
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except Exception as e:                                   # report, do not fail the measurement
        info["power_limit_error"] = str(e)
    return info


def make_input(kind, nbytes):
    import torch
    from conftest import lf_synth_int
    if kind == "lf_synth":
        X, Y = 2048, 2048
        Z = max(1, nbytes // (2 * X * Y))
        t = lf_synth_int((Z, Y, X), 13, seed=1, device="cuda").view(torch.uint8).reshape(-1)[:nbytes]
        return t.cpu().numpy().tobytes()
    return np.random.default_rng(2).integers(0, 256, nbytes, dtype=np.uint8).tobytes()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--mb", type=int, default=256)
    ap.add_argument("--levels", type=int, nargs="+", default=[1, 9])
    ap.add_argument("--kinds", nargs="+", default=["lf_synth", "random"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default="bz2_bench.json")
    a = ap.parse_args()
    import torch
    L = importlib.import_module("lightfieldmicroscopy_pc-bzip2_b200")
    res = {"gpu": gpu_info(), "mib": a.mb, "reps": a.reps, "unit": "GB/s of input (1e9 B/s)", "runs": []}
    for kind in a.kinds:
        data = make_input(kind, a.mb << 20)
        dev = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        for level in a.levels:
            t0 = time.perf_counter(); want = bz2.compress(data, level); t_cpu = time.perf_counter() - t0
            got = L.bz2_compress(data, level)
            if got != want:
                raise SystemExit("%s level %d: GPU stream differs from bz2.compress (%d vs %d bytes)" % (kind, level, len(got), len(want)))
            st = L.stats()
            stages = {k: round(getattr(st, k), 3) for k in ("ms_rle", "ms_bwt", "ms_mtf", "ms_huff", "ms_h2d", "ms_d2h", "ms_total")}
            p = C.c_void_p(); n = C.c_uint64()
            dev_s, host_s = [], []
            for _ in range(a.reps + 1):                      # the first round warms the workspace up and is dropped
                t0 = time.perf_counter()
                rc = L.lib.lfmBz2CompressDevice(dev.data_ptr(), dev.numel(), level, C.byref(p), C.byref(n))
                dev_s.append(time.perf_counter() - t0)
                assert rc == 0 and n.value == len(want)
                dst = L.stats()
                t0 = time.perf_counter(); L.bz2_compress(data, level); host_s.append(time.perf_counter() - t0)
            dev_t, host_t = float(np.median(dev_s[1:])), float(np.median(host_s[1:]))
            t0 = time.perf_counter(); bz2.decompress(want); t_cpu_d = time.perf_counter() - t0
            if L.bz2_decompress(want) != data:
                raise SystemExit("%s level %d: GPU decompression differs from the input" % (kind, level))
            zdev = torch.frombuffer(bytearray(want), dtype=torch.uint8).cuda()
            out = torch.empty(len(data), dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            ddev_s, dhost_s = [], []
            for _ in range(a.reps + 1):
                t0 = time.perf_counter()
                rc = L.lib.lfmBz2DecompressDevice(zdev.data_ptr(), zdev.numel(), out.data_ptr(), out.numel(), C.byref(n))
                ddev_s.append(time.perf_counter() - t0)
                assert rc == 0 and n.value == len(data)
                dd = L.stats()
                t0 = time.perf_counter(); L.bz2_decompress(want); dhost_s.append(time.perf_counter() - t0)
            ddev_t, dhost_t = float(np.median(ddev_s[1:])), float(np.median(dhost_s[1:]))
            dec = {"decompress_device_gbps": round(len(data) / ddev_t / 1e9, 3), "decompress_host_gbps": round(len(data) / dhost_t / 1e9, 3),
                   "python_bz2_decompress_single_core_gbps": round(len(data) / t_cpu_d / 1e9, 4),
                   "decompress_stage_ms_device_call": {"ms_decode": round(dd.ms_decode, 3), "ms_unrle": round(dd.ms_unrle, 3)}}
            dstages = {k: round(getattr(dst, k), 3) for k in ("ms_rle", "ms_bwt", "ms_mtf", "ms_huff")}
            run = {"kind": kind, "level": level, "bytes": len(data), "stream_bytes": len(want), "ratio": round(len(data) / len(want), 4),
                   "compress_device_gbps": round(len(data) / dev_t / 1e9, 3), "compress_host_gbps": round(len(data) / host_t / 1e9, 3),
                   "python_bz2_single_core_gbps": round(len(data) / t_cpu / 1e9, 4),
                   "device_ms": round(dev_t * 1e3, 2), "host_ms": round(host_t * 1e3, 2), "python_bz2_ms": round(t_cpu * 1e3, 1),
                   "stage_ms_device_call": dstages, "dominant_stage": max(dstages, key=dstages.get), "stage_ms_host_call": stages,
                   "gpu_launches": dst.gpu_launches, **dec}
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
