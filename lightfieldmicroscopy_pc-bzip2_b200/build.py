#!/usr/bin/env python3
"""Build liblfm_b200.so (the C-ABI shared library: sm_100a CUDA kernels + C++ host layer) in-tree with nvcc."""
import os, subprocess, sys, hashlib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "liblfm_b200.so")
CU = ["bz_bwt.cu", "bz_encode.cu", "bz_decode.cu", "bz_stream.cu", "lfm_predict.cu", "lfm_select.cu", "lfm_roi.cu", "engine.cu"]
CPP = ["klb_imageHeader.cpp", "klb_ROI.cpp", "klb_imageIO.cpp", "klb_Cwrapper.cpp"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]

def _stamp():
    h = hashlib.sha1()
    for d in (CSRC, os.path.join(ROOT, "include")):
        for f in sorted(os.listdir(d)):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()

def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    stamp_file = os.path.join(HERE, "build", "stamp")
    stamp = _stamp()
    if not force and os.path.exists(OUT) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return OUT
    if not os.path.exists(nvcc):
        if os.path.exists(OUT):
            return OUT                      # GPU box without toolchain changes: use the shipped library
        raise RuntimeError("nvcc not found and no prebuilt liblfm_b200.so")
    bdir = os.path.join(HERE, "build"); os.makedirs(bdir, exist_ok=True)
    inc = ["-I", os.path.join(ROOT, "include"), "-I", CSRC]
    common = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default"]
    procs = []
    objs = []
    for f in CU + CPP:
        o = os.path.join(bdir, f + ".o"); objs.append(o)
        cmd = [nvcc] + ARCH + common + inc + (["-x", "cu"] if f.endswith(".cu") else []) + ["-c", os.path.join(CSRC, f), "-o", o]
        procs.append((f, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    bad = False
    for f, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            bad = True; sys.stderr.write("== %s ==\n%s\n" % (f, out))
        elif verbose and out.strip():
            print("== %s ==\n%s" % (f, out))
    if bad:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc] + ARCH + ["-shared", "-o", OUT] + objs
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout); raise RuntimeError("link failed")
    open(stamp_file, "w").write(stamp)
    return OUT

if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
