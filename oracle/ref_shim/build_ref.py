#!/usr/bin/env python3
"""Builds oracle/_ref/libref_caffe.so: the REFERENCE's own layer sources, compiled where they lie.

TEST INFRASTRUCTURE ONLY (nothing under flownet2_b200/ may load the result).

    python oracle/ref_shim/build_ref.py [--force]

* Sources are compiled straight from /root/reference (never copied); objects, the generated caffe.pb.h and the
  library go to the git-ignored oracle/_ref/ (which DOES travel to the GPU box with the gpurun snapshot).
* The reference's own build system is not run (it needs protobuf, glog, gflags, boost, a CBLAS, OpenCV, HDF5, LMDB,
  none of which exist in the image).  Only those third-party libraries are replaced, by the small stand-ins in
  ref_shim/thirdparty/ (logging macros, std::shared_ptr, <random>, CBLAS prototypes forwarded to the OpenBLAS inside
  the image's scipy wheel) and a generated caffe.pb.h (ref_shim/miniprotoc.py reads the reference's caffe.proto).
  Two reference headers are shadowed (ref_shim/override/): util/io.hpp and the umbrella caffe.hpp, because they
  include boost::filesystem / HDF5 / net / solver.
* Flags follow the reference Makefile (:324,:409-410): -O2 -DNDEBUG, nvcc's default -fmad=true; the arch is sm_100a.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.dirname(HERE)
OUT = os.path.join(ORACLE, "_ref")
GEN = os.path.join(OUT, "gen")
OBJ = os.path.join(OUT, "obj")
LIB = os.path.join(OUT, "libref_caffe.so")
REF = os.environ.get("FN2_REFERENCE", "/root/reference")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

# Reference sources on (or under) the FlowNet2 hot path, SURVEY.md section 8(a) and 8(f).
CORE = ["common.cpp", "syncedmem.cpp", "blob.cpp", "layer.cpp",
        "util/math_functions.cpp", "util/math_functions.cu", "util/im2col.cpp", "util/im2col.cu",
        "util/rng.cpp", "util/benchmark.cpp"]
LAYERS = ["correlation_layer", "correlation_layer1d", "resample_layer", "channel_norm_layer", "flow_warp_layer",
          "data_augmentation_layer", "augmentation_layer_base.cpp",
          "base_conv_layer.cpp", "conv_layer", "deconv_layer", "relu_layer", "neuron_layer.cpp",
          "eltwise_layer", "concat_layer", "slice_layer", "silence_layer",
          "l1loss_layer", "loss_layer.cpp", "power_layer", "input_layer.cpp", "split_layer", "downsample_layer", "flow_augmentation_layer",
          "generate_augmentation_parameters_layer"]

INCLUDES = [os.path.join(HERE, "override"), os.path.join(HERE, "thirdparty"), HERE, GEN,
            os.path.join(REF, "include"), os.path.join(REF, "src"), "/usr/local/cuda/include"]
DEFS = ["-DNDEBUG", "-DUSE_OPENCV=0"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def sources():
    out = [os.path.join(REF, "src/caffe", s) for s in CORE]
    for l in LAYERS:
        base = os.path.join(REF, "src/caffe/layers", l)
        if l.endswith(".cpp"):
            out.append(base)
        else:
            for ext in (".cpp", ".cu"):
                if os.path.exists(base + ext):
                    out.append(base + ext)
    out.append(os.path.join(HERE, "ref_capi.cpp"))
    return out


def shim_hash():
    h = hashlib.sha1()
    for root, _, files in sorted(os.walk(HERE)):
        for fn in sorted(files):
            if fn.endswith((".h", ".hpp", ".py", ".cpp")):
                h.update(open(os.path.join(root, fn), "rb").read())
    return h.hexdigest()


def compile_one(args):
    src, shash, force = args
    name = os.path.relpath(src, REF if src.startswith(REF) else HERE).replace("/", "_") + ".o"
    obj = os.path.join(OBJ, name)
    stamp = obj + ".sha1"
    want = hashlib.sha1((shash + open(src, "rb").read().decode("latin1")).encode("latin1")).hexdigest()
    if not force and os.path.exists(obj) and os.path.exists(stamp) and open(stamp).read() == want:
        return obj
    inc = sum((["-I", i] for i in INCLUDES), [])
    if src.endswith(".cu"):
        cmd = [NVCC] + ARCH + ["-O2", "-std=c++14", "-lineinfo", "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fPIC,-fopenmp,-w",
                                "-w"] + DEFS + inc + ["-c", src, "-o", obj]
    else:
        cmd = ["/usr/bin/g++", "-O2", "-std=c++14", "-fPIC", "-fopenmp", "-pthread", "-w"] + DEFS + inc + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("compile failed: %s\n%s\n%s" % (" ".join(cmd), r.stdout[-6000:], r.stderr[-6000:]))
    open(stamp, "w").write(want)
    return obj


def build(force=False, required=True):
    """-> the library path; None when the reference checkout is not readable and required is False."""
    if not os.path.isdir(REF):
        if os.path.exists(LIB):
            return LIB          # GPU box: the prebuilt library travelled with the snapshot
        if not required:
            return None
        raise RuntimeError("reference checkout %s not present and no prebuilt %s" % (REF, LIB))
    os.makedirs(os.path.join(GEN, "caffe/proto"), exist_ok=True)
    os.makedirs(OBJ, exist_ok=True)
    pb = os.path.join(GEN, "caffe/proto/caffe.pb.h")
    subprocess.run([sys.executable, os.path.join(HERE, "miniprotoc.py"), os.path.join(REF, "src/caffe/proto/caffe.proto"), pb + ".tmp"],
                   check=True)
    if not os.path.exists(pb) or open(pb).read() != open(pb + ".tmp").read():
        os.replace(pb + ".tmp", pb)
    else:
        os.remove(pb + ".tmp")
    shash = shim_hash() + hashlib.sha1(open(pb, "rb").read()).hexdigest()
    srcs = sources()
    with ThreadPoolExecutor(max_workers=8) as ex:
        objs = list(ex.map(compile_one, [(s, shash, force) for s in srcs]))
    newest = max(os.path.getmtime(o) for o in objs)
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < newest:
        cmd = [NVCC] + ARCH + ["-shared", "-o", LIB] + objs + ["-ccbin", "/usr/bin/g++", "-Xcompiler", "-fopenmp",
                                                                "-lcublas", "-lcurand", "-ldl", "-Xlinker", "--no-undefined"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout[-6000:], r.stderr[-6000:]))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
