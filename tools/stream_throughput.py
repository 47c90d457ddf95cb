"""Throughput of frames-to-files paths, and the host memory of the native tool's two paths.

Workload: bench.py's synthetic 1920x1080 x 10-frame 10-bit sequence (make_frames(100)), written to a .yuv, all four QPs,
both components.  Legs, alternated within every step so that all see the same machine state:
  a   PartitionPredictor.predict_frames(host_out=...): int8 vectors in pinned host memory, no files
  a'  Handle.predict_stream in this process, writing the 8 PartitionMat .txt files
  b   tools/native/pmp_predict, default path (reads the whole sequence, one pmp_predict_host call per QP, then files)
  c   tools/native/pmp_predict --stream (one pmp_predict_stream call, files written window by window)
CTU/s counts 128x128 CTUs per QP: frames x (H/64)(W/64)/4 x 4 QPs.  Leg a' also reports its own file-write rate (bytes
over the time spent inside its write callback), which bounds it when the disk is slower than the GPU.
Then the peak resident set of the tool's child process, b and c, on 3840x2160 10-bit sequences of 30 and 60 frames.
The files of b, c and a' must be byte-equal.  Prints one JSON line with the card's name and power limit.

    python tools/stream_throughput.py [--steps 3] [--rss-frames 30,60] [--out-dir DIR]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
COMPS = ("Luma", "Chroma")


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rss-frames", default="30,60", help="4K frame counts of the RSS legs (empty: skip them)")
    ap.add_argument("--out-dir", default=None, help="where the sequences and files go (default: a temporary directory)")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stream_throughput.py needs a CUDA device (no CPU fallback)")
    with tempfile.TemporaryDirectory(prefix="pmp_stream_") as tmp:
        run(args, args.out_dir or tmp)


def write_yuv(path, y, u, v):
    with open(path, "wb") as fp:
        for f in range(y.shape[0]):
            fp.write(y[f].tobytes()); fp.write(u[f].tobytes()); fp.write(v[f].tobytes())


def same_files(d1, d2, names):
    return all(open(os.path.join(d1, n), "rb").read() == open(os.path.join(d2, n), "rb").read() for n in names)


def tool_run(cmd):
    """(seconds, peak RSS of the child in MiB); raises if the tool fails."""
    with tempfile.TemporaryFile() as log:
        t0 = time.perf_counter()
        p = subprocess.Popen(cmd, stdout=log, stderr=subprocess.STDOUT)
        _, status, ru = os.wait4(p.pid, 0)          # this child's own rusage: ru_maxrss in KiB
        dt = time.perf_counter() - t0
        p.returncode = os.waitstatus_to_exitcode(status)
        if p.returncode != 0:
            log.seek(0)
            raise SystemExit("%s failed (%d):\n%s" % (" ".join(cmd), p.returncode, log.read().decode()))
    return dt, ru.ru_maxrss / 1024.0


def run(args, work):
    import torch
    import bench
    from pmp_vvc_tip2023_b200 import _lib, build, export_weights
    from pmp_vvc_tip2023_b200.Inference_QBD import import_yuv420
    from pmp_vvc_tip2023_b200.netspec import QPS
    from pmp_vvc_tip2023_b200.pipeline import PartitionPredictor

    os.makedirs(work, exist_ok=True)
    models = os.path.join(ROOT, "trained_models")
    wdir = os.path.join(work, "pmpw")
    export_weights.export(models, wdir, missing_bd="seeded")
    tool = build.build_native_tool(os.path.join(work, "pmp_predict"))

    W, H, F = bench.WIDTH, bench.HEIGHT, bench.FRAMES
    y, u, v = bench.make_frames(100)
    name = "bench_%dx%d_10bit" % (W, H)
    seq = os.path.join(work, name + ".yuv")
    write_yuv(seq, y, u, v)
    y, u, v = import_yuv420(seq, W, H, F, 1, is10bit=True)
    hy, hu, hv = (torch.from_numpy(a.view(np.int16)).pin_memory() for a in (y, u, v))

    pp = PartitionPredictor(0, engine="tc", chunk=4800)
    pp.load_pkls(models, qps=QPS, missing_bd="seeded")
    per = 2 * (H // 64 * 16) * (W // 64 * 16) + (H // 64 * 8) * (W // 64 * 8) + 3 * (H // 64 * 16) * (W // 64 * 16)
    py_out = {(c, qp): torch.empty((F, per), dtype=torch.int8).pin_memory() for c in COMPS for qp in QPS}
    h = _lib.Handle(0)
    rows = [[h.weights_load(os.path.join(wdir, "%s_%s_%d.pmpw" % (c, t, qp)))[1] for c in COMPS for t in ("Q", "BD")]
            for qp in QPS]
    files = ["%s_%s_QP%d_PartitionMat.txt" % (name, c, qp) for qp in QPS for c in COMPS]
    dirs = {k: os.path.join(work, k) for k in ("a1", "b", "c")}
    write_time = [0.0, 0]          # seconds inside a' write callbacks, bytes written

    def leg_a():
        pp.predict_frames(hy, hu, hv, qps=QPS, host_out=py_out)
        pp.synchronize()

    def leg_a1():
        os.makedirs(dirs["a1"], exist_ok=True)
        fps = [open(os.path.join(dirs["a1"], n), "wb") for n in files]

        def read(f0, nf, yy, uu, vv):
            yy[...] = y[f0:f0 + nf]
            uu[...] = u[f0:f0 + nf]
            vv[...] = v[f0:f0 + nf]

        def write(w):
            t0 = time.perf_counter()
            for q in range(len(QPS)):
                for c in range(2):
                    t = w.text[(q, c)]
                    fps[2 * q + c].write(t)
                    write_time[1] += t.size
            write_time[0] += time.perf_counter() - t0

        h.predict_stream(rows, F, W, H, 2, read, write, outputs=_lib.OUT_TEXT)
        for fp in fps:
            fp.close()

    def leg_tool(key, extra):
        return tool_run([tool, "--input", seq, "--width", str(W), "--height", str(H), "--frames", str(F), "--bitDepth",
                         "10", "--modelDir", wdir, "--outDir", dirs[key]] + extra)

    legs = (("a", leg_a), ("a_prime", leg_a1), ("b", lambda: leg_tool("b", [])),
            ("c", lambda: leg_tool("c", ["--stream"])))
    for _, fn in legs:                  # warm-up: modules, arenas, staging buffers, page cache
        fn()
    write_time[:] = [0.0, 0]
    t = {k: [] for k, _ in legs}
    for _ in range(args.steps):
        for k, fn in legs:
            t0 = time.perf_counter()
            fn()
            t[k].append(time.perf_counter() - t0)
    equal = same_files(dirs["b"], dirs["c"], files) and same_files(dirs["b"], dirs["a1"], files)
    ctus = F * (H // 64) * (W // 64) / 4.0 * len(QPS)
    res = {"workload": "%dx%d x %d frames 10-bit, QPs %s, luma + chroma" % (W, H, F, list(QPS)), "gpu": gpu_info(),
           "steps": args.steps, "files_byte_equal_b_c_a_prime": bool(equal)}
    for k, ts in t.items():
        res[k] = {"ctu_per_s_median": ctus / float(np.median(ts)), "s_per_call": [round(x, 3) for x in ts]}
    res["a_prime_over_a"] = res["a_prime"]["ctu_per_s_median"] / res["a"]["ctu_per_s_median"]
    res["c_over_b"] = res["c"]["ctu_per_s_median"] / res["b"]["ctu_per_s_median"]
    res["a_prime_file_write_MB_per_s"] = write_time[1] / 1e6 / write_time[0] if write_time[0] else None
    h.close()
    pp.close()

    # peak RSS of the tool's two paths on 4K sequences of growing length
    frame_counts = [int(x) for x in args.rss_frames.split(",") if x]
    if frame_counts:
        W4, H4 = 3840, 2160
        y4, u4, v4 = bench.make_frames(101, width=W4, height=H4, frames=max(frame_counts))
        seq4 = os.path.join(work, "rss_%dx%d_10bit.yuv" % (W4, H4))
        write_yuv(seq4, y4, u4, v4)
        del y4, u4, v4
        res["rss_MiB_4k"] = {}
        for nf in frame_counts:
            row = {}
            for key, extra in (("b", []), ("c", ["--stream"])):
                out = os.path.join(work, "rss_" + key)
                dt, rss = tool_run([tool, "--input", seq4, "--width", str(W4), "--height", str(H4), "--frames", str(nf),
                                    "--bitDepth", "10", "--modelDir", wdir, "--outDir", out] + extra)
                row[key] = {"peak_rss_MiB": round(rss, 1), "s": round(dt, 3),
                            "ctu_per_s": nf * (H4 // 64) * (W4 // 64) / 4.0 * len(QPS) / dt}
            names = sorted(os.listdir(os.path.join(work, "rss_b")))
            row["files_byte_equal"] = names == sorted(os.listdir(os.path.join(work, "rss_c"))) and \
                same_files(os.path.join(work, "rss_b"), os.path.join(work, "rss_c"), names)
            equal = equal and row["files_byte_equal"]
            for key in ("b", "c"):
                shutil.rmtree(os.path.join(work, "rss_" + key))
            res["rss_MiB_4k"]["%d_frames" % nf] = row
    print(json.dumps(res))
    if not equal:
        raise SystemExit("the paths wrote different files")


if __name__ == "__main__":
    main()
