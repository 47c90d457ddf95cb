"""Throughput of the Python-free path (pmp_predict_host) next to the Python end-to-end path
(PartitionPredictor.predict_frames with host_out), on the same frames in the same process.

Workload: bench.py's synthetic 1920x1080 x 10-frame 10-bit sequence (written to a .yuv and read back as the native tool
reads it), one QP, both components, chunk 4800.  Both paths start from the same pinned host planes and end with the int8
PartitionMat vectors in pinned host memory; their timed calls alternate so that both see the same machine state.
A third leg times pmp_predict_host on pageable planes and outputs (the native tool's case, staged through the library's
pinned buffers).  Outputs must be byte-equal.  Prints one JSON line with both rates (CTU/s, 128x128 CTUs = 4 blocks per block-QP) and the
card's name and power limit.

    python tools/native_throughput.py [--steps 5] [--qp 32] [--out-dir DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--qp", type=int, default=32)
    ap.add_argument("--chunk", type=int, default=4800)
    ap.add_argument("--out-dir", default=None, help="where the .yuv and the .pmpw files go (default: a temporary directory)")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("native_throughput.py needs a CUDA device (no CPU fallback)")
    with tempfile.TemporaryDirectory(prefix="pmp_native_") as tmp:
        run(args, args.out_dir or tmp)


def run(args, work):
    import torch
    import bench
    from pmp_vvc_tip2023_b200 import _lib, export_weights
    from pmp_vvc_tip2023_b200.Inference_QBD import import_yuv420
    from pmp_vvc_tip2023_b200.pipeline import PartitionPredictor

    os.makedirs(work, exist_ok=True)
    models = os.path.join(ROOT, "trained_models")
    wdir = os.path.join(work, "pmpw")
    export_weights.export(models, wdir, missing_bd="seeded", qps=(args.qp,))

    W, H, F, qp = bench.WIDTH, bench.HEIGHT, bench.FRAMES, args.qp
    y, u, v = bench.make_frames(100)
    seq = os.path.join(work, "bench_%dx%d_10bit.yuv" % (W, H))
    with open(seq, "wb") as fp:
        for f in range(F):
            fp.write(y[f].tobytes()); fp.write(u[f].tobytes()); fp.write(v[f].tobytes())
    y, u, v = import_yuv420(seq, W, H, F, 1, is10bit=True)
    hy, hu, hv = (torch.from_numpy(a.view(np.int16)).pin_memory() for a in (y, u, v))

    pp = PartitionPredictor(0, engine="tc", chunk=args.chunk)
    pp.load_pkls(models, qps=(qp,), missing_bd="seeded")
    per = 2 * (H // 64 * 16) * (W // 64 * 16) + (H // 64 * 8) * (W // 64 * 8) + 3 * (H // 64 * 16) * (W // 64 * 16)
    py_out = {(c, qp): torch.empty((F, per), dtype=torch.int8).pin_memory() for c in ("Luma", "Chroma")}
    h = _lib.Handle(0)
    wsets = [h.weights_load(os.path.join(wdir, "%s_%s_%d.pmpw" % (c, t, qp)))[1] for c in ("Luma", "Chroma")
             for t in ("Q", "BD")]
    nat_out = tuple(torch.empty((F, per), dtype=torch.int8).pin_memory() for _ in range(2))
    nat_pageable = tuple(np.empty((F, per), np.int8) for _ in range(2))

    def run_python():
        pp.predict_frames(hy, hu, hv, qps=(qp,), host_out=py_out)
        pp.synchronize()

    def run_native():
        h.predict_host(wsets, hy, hu, hv, chunk=args.chunk, outs=nat_out)

    def run_native_pageable():          # the native tool's case: pageable planes and outputs, staged by the library
        h.predict_host(wsets, y, u, v, chunk=args.chunk, outs=nat_pageable)

    for _ in range(2):                              # warm-up: modules, arenas, staging buffers
        run_python()
        run_native()
        run_native_pageable()

    def equal_outputs():
        return all(torch.equal(py_out[(c, qp)], nat_out[i]) and np.array_equal(py_out[(c, qp)].numpy(), nat_pageable[i])
                   for i, c in enumerate(("Luma", "Chroma")))

    equal = equal_outputs()
    t = {"python": [], "native": [], "native_pageable": []}
    for _ in range(args.steps):
        for name, fn in (("native", run_native), ("python", run_python), ("native_pageable", run_native_pageable)):
            t0 = time.perf_counter()
            fn()
            t[name].append(time.perf_counter() - t0)
    equal = equal and equal_outputs()
    ctus = F * (H // 64) * (W // 64) / 4.0
    res = {"workload": "%dx%d x %d frames 10-bit, QP %d, luma + chroma, chunk %d" % (W, H, F, qp, args.chunk),
           "gpu": gpu_info(), "steps": args.steps, "outputs_byte_equal": bool(equal)}
    for name, ts in t.items():
        res[name] = {"ctu_per_s_median": ctus / float(np.median(ts)), "ctu_per_s_min_time": ctus / min(ts),
                     "ms_per_call": [round(1e3 * x, 3) for x in ts]}
    res["native_over_python"] = res["native"]["ctu_per_s_median"] / res["python"]["ctu_per_s_median"]
    print(json.dumps(res))
    h.close()
    pp.close()
    if not equal:
        raise SystemExit("pmp_predict_host and predict_frames disagree")


if __name__ == "__main__":
    main()
