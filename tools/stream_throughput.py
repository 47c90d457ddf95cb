"""Throughput of frames-to-files paths, and the host memory of the native tool's two paths.

Workload: bench.py's synthetic 1920x1080 x 10-frame 10-bit sequence (make_frames(100)), written to a .yuv, all four QPs,
both components.  Legs, alternated within every step so that all see the same machine state:
  a   PartitionPredictor.predict_frames(host_out=...): int8 vectors in pinned host memory, no files
  a'  Handle.predict_stream in this process, writing the 8 PartitionMat .txt files
  b   tools/native/pmp_predict, default path (reads the whole sequence, one pmp_predict_host call per QP, then files)
  c   tools/native/pmp_predict --stream (one pmp_predict_stream call, files written window by window)
and, on that sequence and on the 3840x2160 x 30-frame 10-bit sequence of the RSS legs, the several-handle stream
(frames read from the .yuv file, text only, all four QPs), each leg once writing the 8 files and once with a write
callback that only touches the text bytes:
  stream_1h       Handle.predict_stream (pmp_predict_stream) on one handle
  multi_1h        predict_stream_multi (pmp_predict_stream_multi) with that one handle
  multi_2h_dev0   predict_stream_multi with two handles on device 0
  multi_<n>gpu    with two or more visible GPUs: one handle per GPU, and tool_<n>gpu, pmp_predict --stream --devices
                  0,1,... (files); otherwise recorded as not measured
CTU/s counts 128x128 CTUs per QP: frames x (H/64)(W/64)/4 x 4 QPs.  Leg a' also reports its own file-write rate (bytes
over the time spent inside its write callback), which bounds it when the disk is slower than the GPU; the multi legs
report the share of wall time spent inside their callbacks, which names a host-thread limit if there is one.
Then the peak resident set of the tool's child process, b and c, on 3840x2160 10-bit sequences of 30 and 60 frames.
The files of b, c and a' must be byte-equal, and those of every multi leg equal to stream_1h's.  Prints one JSON line
with every used card's name and power limit.

    python tools/stream_throughput.py [--steps 3] [--rss-frames 30,60] [--multi-4k-frames 30] [--out-dir DIR]
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


def gpu_info(all_cards=False):
    r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    lines = r.stdout.strip().splitlines() if r.returncode == 0 and r.stdout.strip() else ["unknown"]
    return lines if all_cards else lines[0].split(", ", 1)[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--rss-frames", default="30,60", help="4K frame counts of the RSS legs (empty: skip them)")
    ap.add_argument("--multi-4k-frames", type=int, default=30, help="frames of the 4K multi-handle legs (0: skip them)")
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

    legs = [("a", leg_a), ("a_prime", leg_a1), ("b", lambda: leg_tool("b", [])),
            ("c", lambda: leg_tool("c", ["--stream"]))]

    # the several-handle stream: one sequence over 1, 2 and one-per-GPU handles, files or touch-only writes
    ndev = torch.cuda.device_count()
    seqs = {"1080p10": (seq, name, W, H, F)}
    frame_counts = [int(x) for x in args.rss_frames.split(",") if x]
    W4, H4 = 3840, 2160
    name4 = "rss_%dx%d_10bit" % (W4, H4)
    seq4 = os.path.join(work, name4 + ".yuv")
    if frame_counts or args.multi_4k_frames > 0:      # one 4K sequence for the multi legs and the RSS legs
        y4, u4, v4 = bench.make_frames(101, width=W4, height=H4, frames=max(frame_counts + [args.multi_4k_frames]))
        write_yuv(seq4, y4, u4, v4)
        del y4, u4, v4
    if args.multi_4k_frames > 0:
        seqs["4k%d" % args.multi_4k_frames] = (seq4, name4, W4, H4, args.multi_4k_frames)

    def load_rows(hh):
        return [[hh.weights_load(os.path.join(wdir, "%s_%s_%d.pmpw" % (c, t_, qp)))[1] for c in COMPS
                 for t_ in ("Q", "BD")] for qp in QPS]

    h2 = _lib.Handle(0)
    multi = {"stream_1h": None, "multi_1h": [(h, rows)], "multi_2h_dev0": [(h, rows), (h2, load_rows(h2))]}
    if ndev >= 2:
        gpu_hs = [_lib.Handle(d) for d in range(1, ndev)]
        multi["multi_%dgpu" % ndev] = [(h, rows)] + [(g, load_rows(g)) for g in gpu_hs]
    cb_time = {}                        # (seq, leg, mode) -> [seconds inside callbacks per call]
    multi_equal = {}                    # (seq, leg) -> files of every call byte-equal to stream_1h's
    after = {}                          # leg key -> run after each timed call, outside the timing

    def multi_dir(skey, leg):
        return os.path.join(work, "m_%s_%s" % (skey, leg))

    def check_and_drop(skey, leg):
        """Compares the leg's files with stream_1h's and deletes them (the 4K texts are 1.3 GB per leg)."""
        nm = seqs[skey][1]
        names = ["%s_%s_QP%d_PartitionMat.txt" % (nm, c, qp) for qp in QPS for c in COMPS]
        same = same_files(multi_dir(skey, "stream_1h"), multi_dir(skey, leg), names)
        multi_equal[(skey, leg)] = multi_equal.get((skey, leg), True) and same
        shutil.rmtree(multi_dir(skey, leg))

    def leg_multi(skey, leg, mode):
        path, nm, w_, h_, f_ = seqs[skey]
        ysz = w_ * h_ * 2
        fsz = ysz * 3 // 2
        mm = np.memmap(path, dtype=np.uint8, mode="r")
        inside = [0.0]
        fps = []
        if mode == "files":
            d = multi_dir(skey, leg)
            os.makedirs(d, exist_ok=True)
            fps = [open(os.path.join(d, "%s_%s_QP%d_PartitionMat.txt" % (nm, c, qp)), "wb") for qp in QPS for c in COMPS]

        def read(f0, nf, yy, uu, vv):
            t0 = time.perf_counter()
            for k in range(nf):
                b0 = (f0 + k) * fsz
                yy[k].view(np.uint8).reshape(-1)[:] = mm[b0:b0 + ysz]
                uu[k].view(np.uint8).reshape(-1)[:] = mm[b0 + ysz:b0 + ysz * 5 // 4]
                vv[k].view(np.uint8).reshape(-1)[:] = mm[b0 + ysz * 5 // 4:b0 + fsz]
            inside[0] += time.perf_counter() - t0

        def write(wnd):
            t0 = time.perf_counter()
            for q in range(len(QPS)):
                for c in range(2):
                    t_ = wnd.text[(q, c)]
                    if fps:
                        fps[2 * q + c].write(t_)
                    else:
                        int(t_[::4096].sum())       # touch one byte per page
            inside[0] += time.perf_counter() - t0

        if leg == "stream_1h":
            h.predict_stream(rows, f_, w_, h_, 2, read, write, outputs=_lib.OUT_TEXT)
        else:
            hr = multi[leg]
            _lib.predict_stream_multi([x[0] for x in hr], [x[1] for x in hr], f_, w_, h_, 2, read, write,
                                      outputs=_lib.OUT_TEXT)
        for fp in fps:
            fp.close()
        cb_time.setdefault((skey, leg, mode), []).append(inside[0])

    def leg_tool_multi(skey):
        path, nm, w_, h_, f_ = seqs[skey]
        return tool_run([tool, "--input", path, "--width", str(w_), "--height", str(h_), "--frames", str(f_), "--bitDepth",
                         "10", "--modelDir", wdir, "--outDir", multi_dir(skey, "tool_%dgpu" % ndev),
                         "--stream", "--devices", ",".join(str(d) for d in range(ndev))])

    for skey in seqs:
        for leg in multi:               # stream_1h first: the others' files are compared with its files
            for mode in ("files", "touch"):
                legs.append(((skey, leg, mode), lambda s_=skey, l_=leg, m_=mode: leg_multi(s_, l_, m_)))
                if mode == "files" and leg != "stream_1h":
                    after[(skey, leg, mode)] = lambda s_=skey, l_=leg: check_and_drop(s_, l_)
        if ndev >= 2:
            key = (skey, "tool_%dgpu" % ndev, "files")
            legs.append((key, lambda s_=skey: leg_tool_multi(s_)))
            after[key] = lambda s_=skey: check_and_drop(s_, "tool_%dgpu" % ndev)

    for k, fn in legs:                  # warm-up: modules, arenas, staging buffers, page cache
        fn()
        if k in after:
            after[k]()
    write_time[:] = [0.0, 0]
    cb_time.clear()
    t = {k: [] for k, _ in legs}
    for _ in range(args.steps):
        for k, fn in legs:
            t0 = time.perf_counter()
            fn()
            t[k].append(time.perf_counter() - t0)
            if k in after:
                after[k]()
    equal = same_files(dirs["b"], dirs["c"], files) and same_files(dirs["b"], dirs["a1"], files)
    ctus = F * (H // 64) * (W // 64) / 4.0 * len(QPS)
    used = gpu_info(all_cards=True)[:max(ndev, 1)]
    res = {"workload": "%dx%d x %d frames 10-bit, QPs %s, luma + chroma" % (W, H, F, list(QPS)), "gpu": gpu_info(),
           "gpus_used": used, "visible_gpus": ndev, "steps": args.steps, "files_byte_equal_b_c_a_prime": bool(equal)}
    for k, ts in t.items():
        if isinstance(k, tuple):
            continue
        res[k] = {"ctu_per_s_median": ctus / float(np.median(ts)), "s_per_call": [round(x, 3) for x in ts]}
    res["a_prime_over_a"] = res["a_prime"]["ctu_per_s_median"] / res["a"]["ctu_per_s_median"]
    res["c_over_b"] = res["c"]["ctu_per_s_median"] / res["b"]["ctu_per_s_median"]
    res["a_prime_file_write_MB_per_s"] = write_time[1] / 1e6 / write_time[0] if write_time[0] else None

    res["multi"] = {}
    for skey, (_, nm, w_, h_, f_) in seqs.items():
        ctus_s = f_ * (h_ // 64) * (w_ // 64) / 4.0 * len(QPS)
        row = {"workload": "%dx%d x %d frames 10-bit, QPs %s, luma + chroma, text only" % (w_, h_, f_, list(QPS))}
        for leg in list(multi) + (["tool_%dgpu" % ndev] if ndev >= 2 else []):
            out = {"texts_byte_equal_to_stream_1h": multi_equal.get((skey, leg), True)}
            equal = equal and out["texts_byte_equal_to_stream_1h"]
            for mode in ("files", "touch"):
                ts = t.get((skey, leg, mode))
                if ts is None:
                    continue
                m = {"ctu_per_s_median": ctus_s / float(np.median(ts)), "s_per_call": [round(x, 3) for x in ts]}
                if (skey, leg, mode) in cb_time:
                    share = [c / x for c, x in zip(cb_time[(skey, leg, mode)], ts)]
                    m["callback_share_of_wall_median"] = round(float(np.median(share)), 3)
                out[mode] = m
            row[leg] = out
        for mode in ("files", "touch"):
            row["multi_1h_over_stream_1h_" + mode] = (row["multi_1h"][mode]["ctu_per_s_median"] /
                                                     row["stream_1h"][mode]["ctu_per_s_median"])
            row["multi_2h_dev0_over_stream_1h_" + mode] = (row["multi_2h_dev0"][mode]["ctu_per_s_median"] /
                                                          row["stream_1h"][mode]["ctu_per_s_median"])
            key = "multi_%dgpu" % ndev
            if ndev >= 2:
                row[key + "_over_n_times_stream_1h_" + mode] = (row[key][mode]["ctu_per_s_median"] /
                                                               (ndev * row["stream_1h"][mode]["ctu_per_s_median"]))
        if ndev < 2:
            row["multi_ngpu"] = row["tool_ngpu"] = "not measured: %d GPU visible" % ndev
        res["multi"][skey] = row
    for hh, _ in multi.get("multi_%dgpu" % ndev, [])[1:]:
        hh.close()
    h2.close()
    h.close()
    pp.close()

    # peak RSS of the tool's two paths on 4K sequences of growing length
    if frame_counts:
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
