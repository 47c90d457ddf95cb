"""In-tree build of libpmp_b200.so (explicit nvcc, sm_100a only; cross-compiles without a GPU)."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpmp_b200.so")
SOURCES = ["api.cu", "nets.cu", "decode.cu", "conv_simt.cu", "conv_tc.cu"]
# host-level entry points (pmp_weights_load, pmp_predict_host, pmp_predict_stream, pmp_format_texts) on top of the core;
# their pmp_destroy releases the host staging and then runs csrc/api.cu's, which is compiled under another name for that
HOST = os.path.join(HERE, "host")
HOST_SOURCES = ["host_api.cu", "text_batch.cu"]
SOURCE_DEFINES = {"api.cu": ["-Dpmp_destroy=pmp_destroy_core"]}
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(d, f) for d in (CSRC, HOST) for f in os.listdir(d)] + \
        [os.path.join(HERE, "..", "include", "pmp_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a into pmp_vvc_tip2023_b200/libpmp_b200.so."""
    if not force and not stale():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    for d, src in [(CSRC, s) for s in SOURCES] + [(HOST, s) for s in HOST_SOURCES]:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [_nvcc()] + flags + SOURCE_DEFINES.get(src, []) + ["-c", os.path.join(d, src), "-o", obj]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out))
        if verbose and out:
            print(out)
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s" % r.stdout)
    return LIB


def build_native_tool(exe):
    """Compile tools/native/pmp_predict.cpp (C++11, the C header and libpmp_b200.so only) into `exe` with g++, the host
    compiler nvcc itself uses; the executable finds the in-tree library through its rpath."""
    root = os.path.dirname(HERE)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++11", "-O2", "-Wall", "-I" + os.path.join(root, "include"),
           os.path.join(root, "tools", "native", "pmp_predict.cpp"), "-o", exe, "-L" + HERE, "-lpmp_b200",
           "-Wl,-rpath," + HERE]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("%s failed:\n%s" % (" ".join(cmd), r.stdout))
    return exe


if __name__ == "__main__":
    import sys
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))
