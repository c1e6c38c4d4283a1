#!/usr/bin/env python3
"""Device-resident .lfm files: write_stack(CUDA tensor) and read_stack / read_roi(..., device="cuda") against the host round trip
a caller holding a CUDA tensor had before (tensor.cpu().numpy() -> write_stack; read_stack -> torch.from_numpy(...).cuda()).

Workloads: c2 (one 2048^2 frame, Nnum 15, way space), the c3s slice (16 x 2048^2) and full-size c3 (101 x 2048^2), both Nnum 13,
way angle, predictor auto-selected.  Inputs are generated on the GPU (lf_synth_int of tests/conftest.py), files go to /dev/shm.
Before any timing: the file written from the tensor equals the file written from its numpy copy byte for byte, and the stacks
decoded into GPU memory and through the host equal the input.  Each timed call ends synchronised (the engine stream is idle and
the file written when the call returns; the host variants end in a synchronous .cuda() / .cpu()); host clock, one warm-up round,
then the median of --reps rounds, the two variants alternating.  Rates are GB/s of raw uint16 pixels (1e9 B/s).

k_roi_gather (the device ROI crop) is timed in a torch.profiler run of its own with CUDA activities: its mean kernel time per call
and bytes/s for 2 x box bytes of traffic, against the B200's 7.7 TB/s HBM3e data-sheet bandwidth.  Writes one JSON file with the
GPU name and power limit beside the numbers; prints it too.

    python tools/device_io_bench.py --reps 5 --out device_io.json
"""
import argparse
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

HBM_BPS = 7.7e12
# name: (frames, H, W, Nnum, way)
WORKLOADS = {"c2": (1, 2048, 2048, 15, 2), "c3s": (16, 2048, 2048, 13, 1), "c3": (101, 2048, 2048, 13, 1)}


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


def timed_pair(reps, fa, fb):
    """one warm-up round, then `reps` rounds of fa and fb alternating: median seconds of each"""
    ta, tb = [], []
    for i in range(reps + 1):
        t0 = time.perf_counter(); fa(); t1 = time.perf_counter(); fb(); t2 = time.perf_counter()
        if i:
            ta.append(t1 - t0); tb.append(t2 - t1)
    return float(np.median(ta)), float(np.median(tb))


def roi_boxes(F, H, W):
    """(name, lb, ub) in x,y,z,c,t"""
    z0, z1 = F // 10, F - 1 - F // 10
    return [("xz_plane", (0, H // 2, 0, 0, 0), (W - 1, H // 2, F - 1, 0, 0)),
            ("yz_plane", (W // 3, 0, 0, 0, 0), (W // 3, H - 1, F - 1, 0, 0)),
            ("frames_aligned", (0, 0, z0, 0, 0), (W - 1, H - 1, z1, 0, 0)),
            ("frames_unaligned", (1, 0, z0, 0, 0), (W - 2, H - 1, z1, 0, 0))]


def box_bytes(lb, ub):
    return 2 * int(np.prod([ub[i] - lb[i] + 1 for i in range(5)]))


def kernel_profile(L, fn, way, boxes, calls):
    """mean k_roi_gather device time per call for each box, from a torch.profiler run with CUDA activities"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, lb, ub in boxes:
        L.read_roi(fn, lb, ub, way=way, device="cuda")            # warm-up outside the trace
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(calls):
                L.read_roi(fn, lb, ub, way=way, device="cuda")
            torch.cuda.synchronize()
        us, n = 0.0, 0
        for e in prof.key_averages():
            if "k_roi_gather" in e.key:
                us += float(getattr(e, "device_time_total", 0.0) or getattr(e, "cuda_time_total", 0.0))
                n += int(e.count)
        if n == 0:
            raise SystemExit("k_roi_gather not found in the profile of %s" % name)
        per = us / n * 1e-6
        nb = box_bytes(lb, ub)
        out[name] = {"box_bytes": nb, "launches": n, "kernel_us": round(per * 1e6, 2),
                     "traffic_gbps": round(2 * nb / per / 1e9, 1), "share_of_hbm": round(2 * nb / per / HBM_BPS, 3)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS))
    ap.add_argument("--profile-calls", type=int, default=20)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out", default="device_io_bench.json")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import tempfile
    import torch
    from conftest import lf_synth_int
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measures the GPU path")
    L = importlib.import_module("lightfieldmicroscopy_pc-bzip2_b200")
    L.set_devices(0, 1)
    res = {"gpu": gpu_info(), "reps": a.reps, "unit": "GB/s of raw uint16 pixels (1e9 B/s)", "hbm_datasheet_bps": HBM_BPS, "runs": []}
    tmp = tempfile.mkdtemp(prefix="lfm_devio_", dir=a.dir)
    fd, fh = os.path.join(tmp, "dev.lfm"), os.path.join(tmp, "host.lfm")
    try:
        for name in a.workloads:
            F, H, W, nnum, way = WORKLOADS[name]
            t = lf_synth_int((F, H, W), nnum, seed=7, device="cuda")
            raw = t.numel() * 2
            # ---- checks first
            L.write_stack(t, fd, nnum=nnum, way=way)
            wst = L.stats()
            L.write_stack(t.cpu().numpy().view(np.uint16), fh, nnum=nnum, way=way)
            with open(fd, "rb") as f1, open(fh, "rb") as f2:
                if f1.read() != f2.read():
                    raise SystemExit("%s: the file written from the tensor differs from the numpy path's" % name)
            back_dev = L.read_stack(fd, way=way, device="cuda")
            rst = L.stats()
            back_host = torch.from_numpy(L.read_stack(fd, way=way).view(np.int16)).cuda()
            if not (torch.equal(back_dev.view(torch.int16).reshape(t.shape), t) and torch.equal(back_host.reshape(t.shape), t)):
                raise SystemExit("%s: decoded stack differs from the input" % name)
            xz = roi_boxes(F, H, W)[0]
            if not torch.equal(L.read_roi(fd, xz[1], xz[2], way=way, device="cuda").view(torch.int16),
                               torch.from_numpy(L.read_roi(fd, xz[1], xz[2], way=way).view(np.int16)).cuda()):
                raise SystemExit("%s: XZ-plane ROI differs between the device and host reads" % name)
            del back_dev, back_host
            # ---- timings
            w_dev, w_host = timed_pair(a.reps, lambda: L.write_stack(t, fd, nnum=nnum, way=way),
                                       lambda: L.write_stack(t.cpu().numpy().view(np.uint16), fh, nnum=nnum, way=way))
            out = torch.empty(t.shape, dtype=torch.uint16, device="cuda")
            r_dev, r_host = timed_pair(a.reps, lambda: L.read_stack(fd, way=way, out=out),
                                       lambda: torch.from_numpy(L.read_stack(fd, way=way).view(np.int16)).cuda())
            xb = box_bytes(xz[1], xz[2])
            x_dev, x_host = timed_pair(a.reps, lambda: L.read_roi(fd, xz[1], xz[2], way=way, device="cuda"),
                                       lambda: torch.from_numpy(L.read_roi(fd, xz[1], xz[2], way=way).view(np.int16)).cuda())
            run = {"workload": name, "shape_zyx": [F, H, W], "nnum": nnum, "way": way, "raw_bytes": raw,
                   "file_bytes": os.path.getsize(fd), "stored_predictor": wst.predictor,
                   "write_device_gbps": round(raw / w_dev / 1e9, 3), "write_host_roundtrip_gbps": round(raw / w_host / 1e9, 3),
                   "write_device_ms": round(w_dev * 1e3, 2), "write_host_roundtrip_ms": round(w_host * 1e3, 2),
                   "read_device_gbps": round(raw / r_dev / 1e9, 3), "read_host_roundtrip_gbps": round(raw / r_host / 1e9, 3),
                   "read_device_ms": round(r_dev * 1e3, 2), "read_host_roundtrip_ms": round(r_host * 1e3, 2),
                   "xz_plane_bytes": xb, "xz_plane_device_ms": round(x_dev * 1e3, 3), "xz_plane_host_roundtrip_ms": round(x_host * 1e3, 3),
                   "device_write_stats_ms": {k: round(getattr(wst, k), 3) for k in ("ms_select", "ms_h2d", "ms_d2h", "ms_total")},
                   "device_read_stats_ms": {k: round(getattr(rst, k), 3) for k in ("ms_h2d", "ms_d2h", "ms_total")}}
            if name == "c3":
                run["k_roi_gather"] = kernel_profile(L, fd, way, roi_boxes(F, H, W), a.profile_calls)
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
            del t, out
            torch.cuda.empty_cache()
    finally:
        for f in (fd, fh):
            if os.path.exists(f):
                os.remove(f)
        os.rmdir(tmp)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
