#!/usr/bin/env python3
"""bench.py -- throughput of the .lfm compress + decompress hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3s|c4s|c5s] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): synthetic 2048x2048 uint16 light-field frames, Nnum=15, predictor way "space", fixed
predictor 4 + bzip2, 96x96x1 KLB blocks (484 per frame).  One STEP = ONE stack of N frames (N = number of GPUs; at N = 1 this is
exactly configs[1]: one frame) is compressed into ONE .lfm image and decompressed again; metric = raw bytes of the stack /
(t_compress + t_decompress), GB/s of raw uint16.

Multi-GPU (torchrun, one rank per GPU) is the split BASELINE.json:north_star names: the frames (z-slabs = contiguous KLB block-id
and payload ranges) of the ONE stack are partitioned over the ranks, every rank compresses its slabs on its own GPU, the
per-block sizes are all-gathered and prefix-summed into blockOffset[] (the only exchange: 4 bytes per block), and -- in the e2e
leg -- rank 0 writes the header + table while every rank streams its payload to its byte offset of ONE shared file; decoding is
the mirror image (every rank fetches and decodes its byte range).  Per-GPU work is fixed as N grows: scaling = "weak".  The
sharded file is compared (md5) with the file ONE GPU writes for the same stack before anything is timed.

  value     device-resident: lfmCompressDevice -> size exchange -> lfmDecompressDevice on frames already in HBM
  e2e       the reference-facing API with PAGEABLE host buffers and a file on /dev/shm, exactly what the reference arm does
            (test/mainTest_lfmIO.cxx:96-126): N = 1: writeLFMstackEx + readKLBstackInPlace; N > 1: lfmShardCompress + lfmWriteHeader +
            lfmShardWritePayload, then readKLBroiInPlace per rank.  H2D, D2H and file I/O inside the timed region.
  e2e_memory   (N = 1) memory -> memory through lfmCompressToBuffer / lfmDecompressFromMemory with pinned buffers, no file
  auto_select  (N = 1, workloads with a fixed predictor) the same frames with headerVersion 0: predictor picked by the 2-D entropy rule
  roofline  the kernel with the largest device time of the step (from the per-stage CUDA-event times of the engine stream; every
            stage is ONE kernel launch per step): algorithmic bytes of that kernel's interface (DESIGN.md 4) per launch / mean
            launch time; peak = MEASURED_PEAKS.json hbm_gbs
  predictor_roofline  the HBM-bound kernels of the path (forward / inverse predictor) alone on a 32-frame stack, 4 B/px
  cpu_baseline / --impl reference: the UNMODIFIED reference (oracle/_ref, its CUDA predictor + threaded CPU bzip2, all host
            cores) on the same N-frame stack, file on /dev/shm; falls back to the oracle port if oracle/_ref is absent.
Inputs rotate through a pool larger than L2 (24 frame sets = 201 MB per GPU > 126 MB), so no step finds its input in L2.

--steps K sets the number of timed steps of every leg: value, e2e, e2e_memory and auto_select, the round trips of cpu_baseline
(the oracle port, when it stands in, times one quarter frame) and the launches predictor_roofline averages per kernel.
--dump-outputs DIR writes what the last timed step of `value` handed its caller (rank 0's shard on several GPUs) to DIR as .npy:
  decoded.npy                lfmDecompressDevice's output, float32 of the uint16 pixels
  payload.npy                lfmCompressDevice's block streams, float32 of the bytes
  block_offset.npy           its blockOffset[], float64
  stored_header_version.npy  its stored headerVersion, float64
decoded.npy and payload.npy longer than their caps (4M / 8M elements) keep, of their flattened form, the elements at the sorted
indices np.random.default_rng(0).integers(0, n, cap); blockOffset[] (at most 3698 blocks per workload) is kept whole: at most
48 MiB and 30 kB in all.  The inputs are seeded, so two builds run with the same
arguments can be compared file for file.
"""
import argparse
import ctypes as C
import hashlib
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (frames per GPU per step, H, W, Nnum, way, headerVersion, block depth, description)
    "c2": (1, 2048, 2048, 15, 2, 8 + 4, 1, "configs[1]: synthetic 2048x2048 uint16 LF frame per GPU, Nnum=15, space predictor 4 + bzip2, 96x96x1 blocks"),
    "c3s": (16, 2048, 2048, 13, 1, 0, 8, "configs[2] slice: 2048x2048x16 uint16 frames per GPU, Nnum=13, angle predictor, 2-D entropy selection, 96x96x8 blocks"),
    "c4s": (64, 1024, 1024, 13, 0, 0x80, 8, "configs[3] slice: 64 frames per GPU of a 1024x1024 video stack (presented as z, Appendix F.5), Nnum=13, way tiles, video bit + 2-D entropy selection, 96x96x8 blocks"),
    "c5s": (16, 4096, 4096, 13, 0, 0, 8, "configs[4] slice: 4096x4096x16 uint16 frames per GPU, Nnum=13, way tiles, 2-D entropy selection, 96x96x8 blocks (full decode)"),
}
POOL = 24
# DRAM bytes of ONE launch measured by ncu --set full (dram__bytes_read.sum + dram__bytes_write.sum): profiles/ncu_traffic.json
NCU_TRAFFIC = {}
try:
    for _k, _v in json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).items():
        NCU_TRAFFIC[tuple(_k.split(":"))] = _v
except Exception:
    pass


def synth_frames(nframes, H, W, nnum, rank):
    from conftest import lf_synth
    return lf_synth((nframes, H, W), nnum, seed=12345 + rank)


def synth_pool(nframes, H, W, nnum, count, rank):
    """LF-synth v1 (SURVEY.md 8d); one pattern, `count` independent noise realisations (cheap to generate); pageable numpy"""
    base = synth_frames(nframes, H, W, nnum, rank)
    rng = np.random.default_rng(777 + rank)
    pool = [base]
    m = base.astype(np.float32)
    for _ in range(count - 1):
        pool.append(np.clip(np.rint(m + rng.normal(0, 1, m.shape).astype(np.float32) * np.sqrt(np.maximum(m, 1)) * 0.5), 0, 65535).astype(np.uint16))
    return pool


def shm_path(name):
    d = "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"
    return os.path.join(d, name)


class ClockSampler:
    def __init__(self, gpu):
        self.rows = []; self.proc = None; self.gpu = gpu

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                                          "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons}


class DeviceBytes:
    """a device buffer the engine owns, seen by torch through the CUDA array interface (no copy)"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


def dump_outputs(dirname, decoded, d_payload, payload_bytes, block_offset, stored_hv):
    """--dump-outputs (module docstring): the caller-visible results of one device round trip as float .npy files"""
    import torch

    def sample(t, cap):
        """t (device tensor) flattened, or the elements at `cap` seeded sorted indices of it, as a host array"""
        t = t.reshape(-1)
        if t.numel() > cap:
            t = t[torch.from_numpy(np.sort(np.random.default_rng(0).integers(0, t.numel(), cap))).to(t.device)]
        return t.cpu().numpy()

    payload = torch.as_tensor(DeviceBytes(d_payload, payload_bytes), device="cuda")
    out = {"decoded": sample(decoded, 1 << 22).view(np.uint16).astype(np.float32),
           "payload": sample(payload, 1 << 23).astype(np.float32),
           "block_offset": block_offset.astype(np.float64),
           "stored_header_version": np.array([stored_hv], np.float64)}
    os.makedirs(dirname, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ reference arm
def load_reference(way):
    """the real reference (GPU build: its CUDA predictor + threaded CPU bzip2); else its CPU-shim build; else None"""
    for kind in ("gpu", "cpu"):
        so = os.path.join(ROOT, "oracle", "_ref", "liblfmref_%s_way%d.so" % (kind, way))
        if os.path.exists(so):
            try:
                return C.CDLL(so), kind
            except OSError:
                continue
    return None, None


def reference_round_trip(pool, nnum, way, hv, bdepth, steps, warmup, settle=True):
    """time `steps` round trips of the reference's writeImage + readImageFull (test/mainTest_lfmIO.cxx:96-126) on /dev/shm.
    Warm-up: at least `warmup` untimed round trips and (settle) until two consecutive ones agree within 5 % (the reference
    cudaMallocs per call and its first calls pay for context / thread start-up), at most warmup + 6."""
    cores = os.cpu_count() or 1
    lib, kind = load_reference(way)
    tmp = shm_path("lfm_bench_ref_%d.lfm" % os.getpid())
    a0 = pool[0]
    Z, H, W = a0.shape
    raw = a0.nbytes
    xyzct = (C.c_uint32 * 5)(W, H, Z, 1, 1)
    bs = (C.c_uint32 * 5)(96, 96, bdepth, 1, 1)
    tc = td = 0.0
    if lib is not None:
        if kind == "cpu" and (hv & 0x7F) < 8:
            hv = 8 + 4              # the CPU-shim build runs the predictor kernels on one core: keep selection out of it
        out = np.empty_like(a0)

        def one(i):
            a = pool[i % len(pool)]
            shv = C.c_int()
            t0 = time.perf_counter()
            rc = lib.ref_write(a.ctypes.data_as(C.c_void_p), tmp.encode(), xyzct, bs, hv, nnum, -1, C.byref(shv))
            t1 = time.perf_counter()
            rc2 = lib.ref_read_full(tmp.encode(), out.ctypes.data_as(C.c_void_p), -1)
            t2 = time.perf_counter()
            assert rc == 0 and rc2 == 0 and np.array_equal(out, a), "reference round trip failed"
            return t1 - t0, t2 - t1
        nw = 0; last = None
        while True:
            c, d = one(nw); nw += 1
            if nw >= warmup and (not settle or (last is not None and abs((c + d) - last) <= 0.05 * last) or nw >= warmup + 6):
                break
            last = c + d
        for i in range(steps):
            c, d = one(nw + i)
            tc += c; td += d
        os.remove(tmp)
        sample = "%d round trips (after %d warm-up) of a %dx%dx%d stack through the unmodified reference (%s build: %s), %d threads, file on %s" % (
            steps, nw, W, H, Z, kind, "its CUDA predictor on the GPU + threaded CPU bzip2" if kind == "gpu" else "its kernels emulated on one CPU core + threaded CPU bzip2",
            cores, os.path.dirname(tmp))
        return dict(kind="reference", cores=cores, sample=sample, tc=tc, td=td, raw=raw * steps, warmups=nw)
    # oracle port, single thread, bounded sample: a quarter of one frame
    from conftest import Oracle
    ora = Oracle()
    a = np.ascontiguousarray(pool[0][:1, :H // 2, :W // 2])
    t0 = time.perf_counter(); rc, _ = ora.write(a, tmp, 8 + 4, nnum, way); t1 = time.perf_counter()
    rc2, back = ora.read(tmp, a.shape, way); t2 = time.perf_counter()
    assert rc == 0 and rc2 == 0 and np.array_equal(back, a)
    os.remove(tmp)
    return dict(kind="port", cores=1, sample="one %dx%d quarter frame through the oracle port (oracle/_ref absent), 1 thread" % (W // 2, H // 2),
                tc=t1 - t0, td=t2 - t1, raw=a.nbytes, warmups=0)


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    nfr, H, W, nnum, way, hv, bdepth, desc = WORKLOADS[args.workload]
    N = max(world, 1) if args.impl == "ours" else max(args.gpus, 1)
    metric = "compress+decompress round-trip GB/s (raw uint16)"
    config = {"workload": desc, "stack_per_step": "%dx%dx%d uint16 (%d frames per GPU x %d GPUs), ONE .lfm image" % (W, H, nfr * N, nfr, N),
              "step": "compress the stack, then decompress it",
              "l2": "inputs rotate through a %d-set pool (%.0f MB per GPU) larger than the 126 MB L2" % (POOL, POOL * nfr * H * W * 2 / 1e6),
              "sharding": "frames (z-slabs: contiguous KLB block-id / payload ranges) of the one stack partitioned over the ranks; only exchange: "
                          "all-gather of the per-block sizes + host prefix sum -> blockOffset[]; e2e: one shared file, pwrite / pread at offsets"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # the same N-frame stack, all host cores (rank 0 alone)
        pool = [np.concatenate([synth_pool(nfr, H, W, nnum, 1, r)[0] for r in range(N)])]
        rng = np.random.default_rng(4242)
        for _ in range(3):
            m = pool[0].astype(np.float32)
            pool.append(np.clip(np.rint(m + rng.normal(0, 1, m.shape).astype(np.float32) * np.sqrt(np.maximum(m, 1)) * 0.5), 0, 65535).astype(np.uint16))
        r = reference_round_trip(pool, nnum, way, hv, bdepth, args.steps, args.warmup)
        val = r["raw"] / (r["tc"] + r["td"]) / 1e9
        line = {"impl": "reference", "metric": metric, "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": r["warmups"],
                "ms_per_step": (r["tc"] + r["td"]) / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u16", "data": "synthetic", "config": config,
                "compress_gbs": r["raw"] / r["tc"] / 1e9, "decompress_gbs": r["raw"] / r["td"] / 1e9,
                "cpu_baseline": {"value": val, "unit": "GB/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = importlib.import_module("lightfieldmicroscopy_pc-bzip2_b200")
    L.set_devices(local, 1)
    L.set_way(way)
    pool = synth_pool(nfr, H, W, nnum, POOL, rank)                       # this rank's frames of every stack of the pool
    dpool = [torch.from_numpy(a.view(np.int16)).cuda() for a in pool]
    raw = pool[0].nbytes                                                 # per rank and step
    bsz = L._u32x5(96, 96, bdepth, 1, 1)
    bsp = C.cast(bsz, C.c_void_p)
    xyzct = L._u32x5(W, H, nfr, 1, 1)                                    # this rank's slabs as a stack of their own
    xyzct_all = L._u32x5(W, H, nfr * world, 1, 1)
    nb = L.lib.lfmNumBlocks(xyzct, bsp)                                  # blocks per rank
    off = np.zeros(nb, np.uint64)
    dout = torch.empty_like(dpool[0])
    shv = C.c_uint8(); dp = C.c_void_p(); pb = C.c_uint64()
    video = hv & 0x80
    auto = (hv & 0x7F) < 8

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def agree_on_predictor(d_frame0):
        """auto-selection: the owner of frame 0 selects, everybody gets the 3 bits (src/klb_imageIO.cpp:2316-2377)"""
        k = torch.zeros(1, dtype=torch.int32, device="cuda")
        if rank == 0:
            kk = C.c_int()
            assert L.lib.lfmSelectDevice(d_frame0, (C.c_uint32 * 2)(W, H), nnum, C.byref(kk), None) == 0
            k[0] = kk.value
        dist.broadcast(k, src=0)
        return int(k[0])

    def exchange_sizes(local_ends):
        """all-gather of the per-block sizes (4 bytes per block) + host prefix sum: blockOffset[] of the whole stack"""
        sizes = np.diff(np.concatenate([[0], local_ends.astype(np.int64)]))
        if world == 1:
            return np.cumsum(sizes).astype(np.uint64)
        mine = torch.from_numpy(sizes.astype(np.int32)).cuda()
        allg = torch.empty(nb * world, dtype=torch.int32, device="cuda")
        dist.all_gather_into_tensor(allg, mine)
        return np.cumsum(allg.cpu().numpy().astype(np.int64)).astype(np.uint64)

    acc = dict(tc=0.0, td=0.0, pred=0.0, sel=0.0, bwt=0.0, rle=0.0, mtf=0.0, huff=0.0, dec=0.0, imtf=0.0, ibwt=0.0, unrle=0.0, unpred=0.0, launches=0, payload=0)

    def step_device(i, timed):
        d = dpool[i % POOL]
        t0 = time.perf_counter()
        hv_i = hv
        sel_ms = 0.0
        if auto and world > 1:
            hv_i = video | (8 + agree_on_predictor(d.data_ptr()))
            sel_ms = L.stats().ms_select if rank == 0 else 0.0
        rc = L.lib.lfmCompressDevice(d.data_ptr(), xyzct, bsp, hv_i, nnum, C.byref(shv), off.ctypes.data, nb, C.byref(dp), C.byref(pb))
        assert rc == 0, "lfmCompressDevice rc=%d %s" % (rc, L.lib.lfmLastError())
        sc = L.stats()
        block_offset = exchange_sizes(off)                       # blockOffset[] of the whole stack (what the header holds)
        t1 = time.perf_counter()
        # decode: every rank takes its range of the table back out
        base = int(block_offset[rank * nb - 1]) if rank else 0
        mine = (block_offset[rank * nb:(rank + 1) * nb] - np.uint64(base)).astype(np.uint64)
        rc = L.lib.lfmDecompressDevice(dp, mine.ctypes.data, nb, xyzct, bsp, shv.value, nnum, dout.data_ptr())
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        assert rc == 0, "lfmDecompressDevice rc=%d" % rc
        sd = L.stats()
        if timed:
            acc["tc"] += t1 - t0; acc["td"] += t2 - t1
            acc["pred"] += sc.ms_predict; acc["sel"] += sc.ms_select + sel_ms; acc["unpred"] += sd.ms_unpredict; acc["bwt"] += sc.ms_bwt; acc["rle"] += sc.ms_rle; acc["mtf"] += sc.ms_mtf; acc["huff"] += sc.ms_huff
            acc["dec"] += sd.ms_decode; acc["imtf"] += sd.ms_imtf; acc["ibwt"] += sd.ms_ibwt; acc["unrle"] += sd.ms_unrle
            acc["launches"] += sc.gpu_launches + sd.gpu_launches + (12 if (auto and world > 1 and rank == 0) else 0); acc["payload"] += pb.value
        return d

    for i in range(args.warmup):
        d = step_device(i, False)
    assert torch.equal(dout, d), "device round trip mismatch"
    sampler = ClockSampler(local); sampler.start()
    barrier()
    t_start = time.perf_counter()
    for i in range(args.steps):
        step_device(args.warmup + i, True)
    barrier(); t_all = time.perf_counter() - t_start
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:                   # before the next engine call releases the payload
        dump_outputs(args.dump_outputs, dout, dp.value, pb.value, off, shv.value)

    # ---- e2e: the reference-facing API, PAGEABLE host buffers, ONE file on /dev/shm (what the reference arm does)
    fname = shm_path("lfm_bench_%s_%d.lfm" % (os.environ.get("MASTER_PORT", "single"), os.getppid() if world > 1 else os.getpid()))
    if world > 1:                                     # all ranks must name the same file
        obj = [fname]
        dist.broadcast_object_list(obj, src=0)
        fname = obj[0]
    hout = np.empty_like(pool[0])                     # pageable
    e2e = dict(tc=0.0, td=0.0, h2d=0, d2h=0, file=0)
    trace = []
    lb = L._u32x5(0, 0, rank * nfr, 0, 0); ub = L._u32x5(W - 1, H - 1, (rank + 1) * nfr - 1, 0, 0)
    hdr_bytes = 320 + 8 * nb * world

    def step_e2e(i, timed, check=False):
        a = pool[i % POOL]
        t0 = time.perf_counter()
        if world == 1:
            rc = L.lib.writeLFMstackEx(a.ctypes.data, os.fsencode(fname), xyzct, 1, -1, None, bsp, 1, None, hv, nnum)
            assert rc == 0, "writeLFMstackEx rc=%d" % rc
            nfile = os.path.getsize(fname) if (timed or check) else 0
            t1 = time.perf_counter()
            dt = C.c_int()
            rc = L.lib.readKLBstackInPlace(os.fsencode(fname), hout.ctypes.data, C.byref(dt), -1)
            assert rc == 0, "readKLBstackInPlace rc=%d" % rc
            t2 = time.perf_counter()
            npay = nfile - hdr_bytes
        else:
            hv_i = hv
            if auto:
                d0 = torch.from_numpy(a[0].view(np.int16)).cuda() if rank == 0 else None
                hv_i = video | (8 + agree_on_predictor(d0.data_ptr() if rank == 0 else 0))
            stored, sizes, npay = L.shard_compress(a, hv_i, nnum=nnum, block_size=(96, 96, bdepth, 1, 1))
            ta = time.perf_counter()
            block_offset = exchange_sizes(np.cumsum(sizes.astype(np.int64)))
            tb = time.perf_counter()
            if rank == 0:
                L.write_header(fname, (W, H, nfr * world, 1, 1), (96, 96, bdepth, 1, 1), stored, nnum, block_offset)
            tc = time.perf_counter()
            L.shard_write_payload(fname, hdr_bytes + (int(block_offset[rank * nb - 1]) if rank else 0))
            td = time.perf_counter()
            dist.barrier()                             # the file is complete
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if timed and os.environ.get("LFM_BENCH_TRACE"):
                trace.append((ta - t0, tb - ta, tc - tb, td - tc, t1 - td))
            rc = L.lib.readKLBroiInPlace(os.fsencode(fname), hout.ctypes.data, lb, ub, -1)
            assert rc == 0, "readKLBroiInPlace rc=%d" % rc
            t2 = time.perf_counter()
        if check:
            assert np.array_equal(hout, a), "e2e round trip mismatch"
        if timed:
            e2e["tc"] += t1 - t0; e2e["td"] += t2 - t1
            e2e["h2d"] += a.nbytes + npay; e2e["d2h"] += npay + a.nbytes; e2e["file"] += 2 * npay
        return npay

    # before anything is timed: the sharded file must be byte-identical to the file ONE GPU writes for the same stack
    sharded_file_md5 = None
    step_e2e(0, False, check=True)
    if world > 1:
        if rank == 0:
            sharded_file_md5 = hashlib.md5(open(fname, "rb").read()).hexdigest()
            whole = np.concatenate([pool[0]] + [synth_frames(nfr, H, W, nnum, r) for r in range(1, world)])
            single = shm_path("lfm_bench_single_%d.lfm" % os.getpid())
            L.write_stack(whole, single, header_version=hv, nnum=nnum, block_size=(96, 96, bdepth, 1, 1))
            single_md5 = hashlib.md5(open(single, "rb").read()).hexdigest()
            os.remove(single)
            assert sharded_file_md5 == single_md5, "the file written by %d ranks differs from the single-GPU file of the same stack" % world
        barrier()
    step_e2e(1, False, check=True)
    barrier()
    te0 = time.perf_counter()
    for i in range(args.steps):
        step_e2e(2 + i, True)
    barrier(); t_e2e = time.perf_counter() - te0
    if trace:                                              # LFM_BENCH_TRACE=1: where the sharded write spends its time, per rank (stderr)
        m = np.mean(np.array(trace), axis=0) * 1e3
        sys.stderr.write("rank %d e2e write: shard_compress %.3f | size exchange %.3f | header %.3f | payload -> file %.3f | barrier %.3f ms\n" % ((rank,) + tuple(m)))
    if rank == 0 and os.path.exists(fname):
        os.remove(fname)

    # ---- (N = 1) memory -> memory with pinned buffers, no file: lfmCompressToBuffer / lfmDecompressFromMemory
    e2m = None
    if world == 1:
        EP = 4
        hin = [torch.from_numpy(pool[i].view(np.int16)).pin_memory() for i in range(EP)]
        hin_np = [t.numpy().view(np.uint16) for t in hin]
        hblob = torch.empty(raw + raw // 2 + (1 << 20), dtype=torch.uint8).pin_memory(); hblob_np = hblob.numpy()
        hpin = torch.empty_like(hin[0]).pin_memory(); hpin_np = hpin.numpy().view(np.uint16)
        e2m = dict(tc=0.0, td=0.0)
        for i in range(2 + args.steps):
            a = hin_np[i % EP]
            t0 = time.perf_counter()
            nblob = L.compress_into(a, hblob_np, header_version=hv, nnum=nnum, block_size=(96, 96, bdepth, 1, 1), way=way)
            t1 = time.perf_counter()
            L.decompress_into(hblob_np, nblob, hpin_np, way=way)
            t2 = time.perf_counter()
            if i < 2:
                assert np.array_equal(hpin_np, a), "memory round trip mismatch"
            else:
                e2m["tc"] += t1 - t0; e2m["td"] += t2 - t1

    # ---- the same stack with the predictor chosen by the 2-D entropy rule on frame 0 (headerVersion 0: SURVEY.md 8d asks for C2 both
    # fixed and auto): device resident, a few steps, N = 1 only
    auto_leg = None
    if world == 1 and not auto:
        ta = dict(tc=0.0, td=0.0, sel=0.0, k=-1)
        nst = args.steps
        for i in range(2 + nst):
            d = dpool[i % POOL]
            torch.cuda.synchronize(); t0 = time.perf_counter()
            rc = L.lib.lfmCompressDevice(d.data_ptr(), xyzct, bsp, video, nnum, C.byref(shv), off.ctypes.data, nb, C.byref(dp), C.byref(pb))
            assert rc == 0, "lfmCompressDevice (auto) rc=%d" % rc
            t1 = time.perf_counter()
            sc = L.stats()
            rc = L.lib.lfmDecompressDevice(dp, off.ctypes.data, nb, xyzct, bsp, shv.value, nnum, dout.data_ptr())
            torch.cuda.synchronize(); t2 = time.perf_counter()
            assert rc == 0, "lfmDecompressDevice (auto) rc=%d" % rc
            if i < 2:
                assert torch.equal(dout, d), "auto-select round trip mismatch"
            else:
                ta["tc"] += t1 - t0; ta["td"] += t2 - t1; ta["sel"] += sc.ms_select; ta["k"] = sc.predictor
        auto_leg = {"value": raw * nst / (ta["tc"] + ta["td"]) / 1e9, "unit": "GB/s", "steps": nst, "ms_per_step": (ta["tc"] + ta["td"]) / nst * 1e3,
                    "ms_select": ta["sel"] / nst, "selected_predictor": ta["k"], "headerVersion": int(video),
                    "note": "same frames, predictor picked per stack by the 2-D entropy rule (7 candidate predictions + 8 entropy estimates on frame 0)"}

    # ---- predictor kernels alone (the HBM-bound stage the north star quotes a roofline target for): forward and inverse
    # on a 32-frame 2048x2048 stack (268 MB, larger than L2), algorithmic traffic 4 B/px, timed by CUDA events on the
    # engine stream inside lfmDebugPredictDevice.  Rank 0 only.
    pred_roof = None
    if rank == 0:
        try:
            PF = 32
            big = torch.from_numpy(np.ascontiguousarray(np.tile(pool[0][:1], (PF, 1, 1))).view(np.int16)).cuda()
            big += torch.arange(PF, dtype=torch.int16, device="cuda").view(PF, 1, 1)        # frames differ
            symb = torch.empty_like(big); back = torch.empty_like(big)
            xyz_b = L._u32x5(W, H, PF, 1, 1)
            ms = C.c_float()
            pred_roof = {"stack": "%dx%dx%d uint16 (%.0f MB)" % (W, H, PF, big.numel() * 2 / 1e6), "bytes_per_px": 4, "runs": {}}
            for wy, kk in ((1, 4), (2, 4), (0, 4), (2, 1), (1, 2), (0, 7)):
                L.set_way(wy)
                for inv, src, dst in ((0, big, symb), (1, symb, back)):
                    assert L.lib.lfmDebugPredictDevice(src.data_ptr(), dst.data_ptr(), xyz_b, nnum, kk, 0, inv, 2, C.byref(ms)) == 0
                    assert L.lib.lfmDebugPredictDevice(src.data_ptr(), dst.data_ptr(), xyz_b, nnum, kk, 0, inv, args.steps, C.byref(ms)) == 0
                    gbs = 4.0 * big.numel() / (ms.value * 1e-3) / 1e9
                    pred_roof["runs"]["way%d_k%d_%s" % (wy, kk, "inverse" if inv else "forward")] = {"ms": ms.value, "achieved_gbs": gbs}
                assert torch.equal(back, big), "predictor round trip mismatch"
            L.set_way(way)
            del big, symb, back
        except Exception as ex:
            pred_roof = {"error": repr(ex)}
            L.set_way(way)

    t_step = torch.tensor([t_all, t_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_step, op=dist.ReduceOp.MAX)
    t_max, t_e2e_max = float(t_step[0]), float(t_step[1])
    total_raw = raw * args.steps * world
    value = total_raw / t_max / 1e9
    e2e_value = total_raw / t_e2e_max / 1e9

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        ratio = raw * args.steps / max(acc["payload"], 1)
        n_post_rle = raw                        # LF-synth frames have no long runs: post-RLE1 length == raw length within 0.1 %
        comp = acc["payload"] / args.steps      # compressed bytes per step (this rank)
        stage_ms = {k: acc[k] / args.steps for k in ("sel", "pred", "rle", "bwt", "mtf", "huff", "dec", "imtf", "ibwt", "unrle", "unpred")}
        # kernel behind every block-codec stage and the algorithmic bytes of its interface per launch (DESIGN.md 4):
        # n = run-length coded block bytes (== raw here), comp = compressed bytes
        kernels = {"rle": ("k_rle1", raw + n_post_rle), "bwt": ("k_bwt", 2 * n_post_rle), "mtf": ("k_mtf", 2 * n_post_rle),
                   "huff": ("k_huff_pack", n_post_rle + comp), "dec": ("k_huff_decode", comp + n_post_rle), "imtf": ("k_imtf", 2 * n_post_rle),
                   "ibwt": ("k_inv_bwt", 2 * n_post_rle), "unrle": ("k_unrle", n_post_rle + raw)}
        top = max(kernels, key=lambda k: stage_ms[k])
        kname, kbytes = kernels[top]
        k_ms = stage_ms[top]
        achieved = kbytes / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
        cpu = None
        if world == 1:
            try:
                rb = reference_round_trip(pool[:4], nnum, way, hv, bdepth, args.steps, 2, settle=False)
                cpu = {"value": rb["raw"] / (rb["tc"] + rb["td"]) / 1e9, "unit": "GB/s", "cores": rb["cores"], "kind": rb["kind"], "sample": rb["sample"],
                       "compress_gbs": rb["raw"] / rb["tc"] / 1e9, "decompress_gbs": rb["raw"] / rb["td"] / 1e9}
            except Exception as ex:            # the baseline must never take the bench line down
                cpu = {"value": None, "unit": "GB/s", "cores": os.cpu_count(), "kind": "reference", "sample": "failed: %r" % (ex,)}
        step_ms = t_max / args.steps * 1e3
        line = {"metric": metric, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u16", "data": "synthetic", "config": config,
                "compress_gbs": raw * world * args.steps / acc["tc"] / 1e9, "decompress_gbs": raw * world * args.steps / acc["td"] / 1e9,
                "compression_ratio": ratio, "stage_ms_per_step": stage_ms,
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": e2e["h2d"] // args.steps, "d2h_bytes_per_step": e2e["d2h"] // args.steps,
                        "file_bytes_per_step": e2e["file"] // args.steps,
                        "compress_gbs": raw * world * args.steps / e2e["tc"] / 1e9, "decompress_gbs": raw * world * args.steps / e2e["td"] / 1e9,
                        "api": "writeLFMstackEx + readKLBstackInPlace" if world == 1 else "lfmShardCompress + lfmWriteHeader + lfmShardWritePayload, readKLBroiInPlace per rank",
                        "host_memory": "pageable (numpy)", "file": os.path.dirname(fname), "bytes_are_per_rank": world > 1},
                "gpu_launches": int(acc["launches"]),
                "roofline": {"bound": "hbm", "kernel": "%s (largest device time of the step: %.3f ms of %.3f ms; one launch over the %d KLB blocks of a rank)" % (kname, k_ms, step_ms, nb),
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": NCU_TRAFFIC.get((kname, args.workload)),
                             "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full (profiles/)",
                             "peak_source": peak_src, "algorithmic_bytes_per_launch": kbytes, "launch_ms": k_ms,
                             "per_kernel": {kernels[k][0]: {"ms": stage_ms[k], "achieved_gbs": kernels[k][1] / (stage_ms[k] * 1e-3) / 1e9 if stage_ms[k] > 0 else None} for k in kernels},
                             "note": "the block codec (sort, entropy coding) is latency / shared-memory bound, not HBM bound: the HBM roofline is quoted as the contract asks; the HBM-bound kernels of the path are the predictors, see predictor_roofline"},
                "predictor_roofline": None if pred_roof is None else dict(pred_roof, peak=peak, unit="GB/s",
                    frac={k: v["achieved_gbs"] / peak for k, v in pred_roof.get("runs", {}).items()})}
        if auto_leg is not None:
            line["auto_select"] = auto_leg
        if e2m is not None:
            line["e2e_memory"] = {"value": raw * args.steps / (e2m["tc"] + e2m["td"]) / 1e9, "unit": "GB/s", "api": "lfmCompressToBuffer + lfmDecompressFromMemory, pinned host buffers, no file",
                                  "compress_gbs": raw * args.steps / e2m["tc"] / 1e9, "decompress_gbs": raw * args.steps / e2m["td"] / 1e9}
        if sharded_file_md5 is not None:
            line["sharded_file"] = {"md5": sharded_file_md5, "equals_single_gpu_file": True}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
