"""Cost of a decode-threshold sweep: four settings of lamb1..lamb5 from one net pass against one setting and against four
separate calls.

Workload: the 3840x2160 x 30-frame 10-bit sequence of tools/stream_throughput.py (bench.make_frames(101)), written to a
.yuv and read from it window by window, QP 32, luma + chroma, text only.  Legs, alternated within every step so that
all see the same machine state, each once with a write callback that only touches the text bytes and once writing the
PartitionMat files:
  a  Handle.predict_stream, one row (pmp_predict_stream)
  b  Handle.predict_stream(lamb=...), four rows sharing QP 32's weights with the default thresholds and
     cases.LAMB_SETS a, b, c (pmp_predict_stream_ex: one net pass per window, four decodes)
  c  four one-row pmp_predict_stream_ex calls, one per setting (four net passes)
Reports the median wall time of each leg, b / a and c / a, and the share of the wall time spent inside the callbacks.
Checks that b's row 0 files equal a's and that b's row i files equal c's call i, byte for byte.  Prints one JSON line
with the card's name and power limit.

    python tools/lamb_sweep_throughput.py [--steps 2] [--frames 30] [--out FILE]
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
COMPS = ("Luma", "Chroma")
QP = 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("lamb_sweep_throughput.py needs a CUDA device (no CPU fallback)")
    with tempfile.TemporaryDirectory(prefix="pmp_lamb_") as tmp:
        res = run(args, tmp)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fp:
            fp.write(line + "\n")
    if not res["byte_equal"]["b_row0_equals_a"] or not res["byte_equal"]["b_rows_equal_c_calls"]:
        raise SystemExit("the legs wrote different files")


def run(args, work):
    import bench
    from pmp_vvc_tip2023_b200 import _lib, export_weights, ops
    from tests import cases
    from tools.stream_throughput import gpu_info, same_files, write_yuv

    settings = [tuple(ops.DEFAULT_LAMB)] + [cases.LAMB_SETS[k] for k in ("a", "b", "c")]
    wdir = os.path.join(work, "pmpw")
    export_weights.export(os.path.join(ROOT, "trained_models"), wdir, missing_bd="seeded")
    W, H, F = 3840, 2160, args.frames
    name = "sweep_%dx%d_10bit" % (W, H)
    seq = os.path.join(work, name + ".yuv")
    y, u, v = bench.make_frames(101, width=W, height=H, frames=F)
    write_yuv(seq, y, u, v)
    del y, u, v
    h = _lib.Handle(0)
    row = [h.weights_load(os.path.join(wdir, "%s_%s_%d.pmpw" % (c, t, QP)))[1] for c in COMPS for t in ("Q", "BD")]
    ysz, fsz = W * H * 2, W * H * 3
    mm = np.memmap(seq, dtype=np.uint8, mode="r")
    inside = [0.0]

    def read(f0, nf, yy, uu, vv):
        t0 = time.perf_counter()
        for k in range(nf):
            b0 = (f0 + k) * fsz
            yy[k].view(np.uint8).reshape(-1)[:] = mm[b0:b0 + ysz]
            uu[k].view(np.uint8).reshape(-1)[:] = mm[b0 + ysz:b0 + ysz * 5 // 4]
            vv[k].view(np.uint8).reshape(-1)[:] = mm[b0 + ysz * 5 // 4:b0 + fsz]
        inside[0] += time.perf_counter() - t0

    def writer(fps):
        def write(w):
            t0 = time.perf_counter()
            for (r, c), t in w.text.items():
                if fps:
                    fps[2 * r + c].write(t)
                else:
                    int(t[::4096].sum())        # touch one byte per page
            inside[0] += time.perf_counter() - t0
        return write

    def leg_dir(leg):
        return os.path.join(work, "files_" + leg)

    def names(r):
        return ["row%d_%s_PartitionMat.txt" % (r, c) for c in COMPS]

    def call(leg, lambs, mode, first_row=0):
        """One stream call; lambs None: one row through pmp_predict_stream, else one row per setting."""
        nrows = 1 if lambs is None else len(lambs)
        fps = []
        if mode == "files":
            os.makedirs(leg_dir(leg), exist_ok=True)
            fps = [open(os.path.join(leg_dir(leg), n), "wb") for r in range(first_row, first_row + nrows)
                   for n in names(r)]
        h.predict_stream([row] * nrows, F, W, H, 2, read, writer(fps), outputs=_lib.OUT_TEXT, lamb=lambs)
        for fp in fps:
            fp.close()

    legs = {"a": lambda mode: call("a", None, mode),
            "b": lambda mode: call("b", settings, mode),
            "c": lambda mode: [call("c", [s], mode, first_row=i) for i, s in enumerate(settings)]}
    equal = {"b_row0_equals_a": True, "b_rows_equal_c_calls": True}

    def check_and_drop():
        equal["b_row0_equals_a"] &= same_files(leg_dir("a"), leg_dir("b"), names(0))
        equal["b_rows_equal_c_calls"] &= all(same_files(leg_dir("b"), leg_dir("c"), names(r)) for r in range(4))
        for leg in legs:
            shutil.rmtree(leg_dir(leg))

    times = {(leg, mode): [] for mode in ("touch", "files") for leg in legs}
    cb = {k: [] for k in times}
    for step in range(args.steps + 1):          # step 0 warms up: modules, arena, staging, page cache
        for mode in ("touch", "files"):
            for leg, fn in legs.items():
                inside[0] = 0.0
                t0 = time.perf_counter()
                fn(mode)
                dt = time.perf_counter() - t0
                if step:
                    times[(leg, mode)].append(dt)
                    cb[(leg, mode)].append(inside[0] / dt)
            if mode == "files":
                check_and_drop()
    h.close()
    ctus = F * (H // 64) * (W // 64) / 4.0
    res = {"workload": "%dx%d x %d frames 10-bit, QP %d, luma + chroma, text only" % (W, H, F, QP),
           "gpu": gpu_info(), "steps": args.steps,
           "settings": {"row%d" % i: list(s) for i, s in enumerate(settings)},
           "legs": {"a": "pmp_predict_stream, one row (default thresholds)",
                    "b": "pmp_predict_stream_ex, four rows on QP 32's weights: one net pass, four decodes",
                    "c": "four one-row pmp_predict_stream_ex calls, one per setting"},
           "byte_equal": equal}
    for mode in ("touch", "files"):
        m = {}
        for leg in legs:
            ts = times[(leg, mode)]
            m[leg] = {"s_median": round(float(np.median(ts)), 3), "s_per_call": [round(x, 3) for x in ts],
                      "ctu_per_s_per_setting_median": ctus * (1 if leg == "a" else 4) / float(np.median(ts)),
                      "callback_share_of_wall_median": round(float(np.median(cb[(leg, mode)])), 3)}
        m["b_over_a"] = round(m["b"]["s_median"] / m["a"]["s_median"], 4)
        m["c_over_a"] = round(m["c"]["s_median"] / m["a"]["s_median"], 4)
        res[mode] = m
    return res


if __name__ == "__main__":
    main()
