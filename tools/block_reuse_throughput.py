"""Throughput of the window pipeline's reuse of repeated blocks, and what the grouping costs on content without repeats.

Speed-up: pmp_predict_stream on one handle, all four QPs, text only with a write callback that touches one byte per page
(the touch-only legs of tools/stream_throughput.py), default windows, on 1920x1080 and 3840x2160 x F-frame 10-bit
sequences of four kinds (the generators of tests/test_gpu_block_reuse.py):
  static     frame 0 repeated
  letterbox  black bars 140 rows high at 1080p (280 at 2160p), Y 64, U/V 512
  mixed      natural frames interleaved with repeats
  natural    two synthetic frames, alternated and shifted by 6 more pixels per frame (no block repeats)
Each is timed against its perturbed twin (same shape, every block marked so that all differ; checked with
pmp_block_stats).  Reported: CTU/s of both (128x128 CTUs per QP: frames x (H/64)(W/64)/4 x 4 QPs), the computed / blocks
fraction and the ratio.

Overhead (--parent-lib FILE: another build of libpmp_b200.so, e.g. the parent commit's): the 3840x2160 x F natural
sequence through the 4K legs of tools/stream_throughput.py, pmp_predict_stream on one handle (stream_1h) and
pmp_predict_stream_multi with two handles on device 0 (multi_2h_dev0), touch-only writes, alternating the two builds
within every step; both builds are loaded into this process, each with its own handles.  The spread is max - min over the
steps of one (build, leg).

Grouping share: CUDA events around pmp_debug_block_groups on one default 4K window's cut blocks (luma and chroma,
64-bit fingerprints), next to that window's share of the stream_1h time.

Prints one JSON line with the card's name and power limit, read in the same run.

    python tools/block_reuse_throughput.py [--steps 3] [--frames 30] [--parent-lib FILE] [--out FILE]
"""
import argparse
import ctypes
import json
import os
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


def natural(width, height, frames, seed):
    from pmp_vvc_tip2023_b200 import synth
    y, u, v = synth.synth_yuv420(width, height, 2, seed=seed)
    return (np.stack([np.roll(y[i % 2], 6 * i, axis=1) for i in range(frames)]),
            np.stack([np.roll(u[i % 2], 3 * i, axis=1) for i in range(frames)]),
            np.stack([np.roll(v[i % 2], 3 * i, axis=1) for i in range(frames)]))


def sequence(kind, base):
    y, u, v = base
    f, height = y.shape[0], y.shape[1]
    if kind == "natural":
        return y, u, v
    if kind == "static":
        return tuple(np.repeat(a[:1], f, 0) for a in (y, u, v))
    if kind == "letterbox":
        y, u, v = y.copy(), u.copy(), v.copy()
        bar = 2 * round(70 * height / 1080)
        y[:, :bar], y[:, height - bar:] = 64, 64
        for c in (u, v):
            c[:, :bar // 2], c[:, (height - bar) // 2:] = 512, 512
        return y, u, v
    if kind == "mixed":
        idx = [i - 1 if i % 3 == 1 else i for i in range(f)]        # every third frame repeats the previous one
        return tuple(np.ascontiguousarray(a[idx]) for a in (y, u, v))
    raise KeyError(kind)


def perturbed(y, u, v):
    """Every block of every frame marked in two luma samples and one U and one V sample: no two blocks are equal."""
    y, u, v = y.copy(), u.copy(), v.copy()
    f, hgt, wid = y.shape
    bh, bw = hgt // 64, wid // 64
    for i in range(bh):
        for j in range(bw):
            k = (np.arange(f) * bh + i) * bw + j
            lo, hi = (k % 256) * 4, (k // 256 % 256) * 4
            y[:, 64 * i + 30, 64 * j + 30], y[:, 64 * i + 31, 64 * j + 30] = lo, hi
            u[:, 32 * i + 15, 32 * j + 15], v[:, 32 * i + 15, 32 * j + 15] = lo, hi
    return y, u, v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--parent-lib", default=None, help="another build of libpmp_b200.so for the overhead legs")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("block_reuse_throughput.py needs a CUDA device (no CPU fallback)")
    with tempfile.TemporaryDirectory(prefix="pmp_reuse_") as tmp:
        res = run(args, tmp)
    res["gpu"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fp:
            fp.write(line + "\n")


def run(args, work):
    import torch
    from pmp_vvc_tip2023_b200 import _lib, export_weights, ops
    from pmp_vvc_tip2023_b200.netspec import QPS

    wdir = os.path.join(work, "pmpw")
    export_weights.export(os.path.join(ROOT, "trained_models"), wdir, missing_bd="seeded")
    libs = {"this": _lib.lib()}
    if args.parent_lib:
        libs["parent"] = ctypes.CDLL(os.path.abspath(args.parent_lib))
        for name, (rt, at) in _lib.SIGNATURES.items():
            if hasattr(libs["parent"], name):
                fn = getattr(libs["parent"], name)
                fn.restype, fn.argtypes = rt, at

    def use(which):                 # route the binding's calls to one build
        _lib._lib = libs[which]

    def handle():
        h = _lib.Handle(0)
        rows = [[h.weights_load(os.path.join(wdir, "%s_%s_%d.pmpw" % (c, t, qp)))[1] for c in COMPS for t in ("Q", "BD")]
                for qp in QPS]
        return h, rows

    use("this")
    h, rows = handle()

    def stream(hs, rws, seq, wid, hgt):
        y, u, v = seq
        f = y.shape[0]

        def read(f0, nf, yy, uu, vv):
            yy[...] = y[f0:f0 + nf]
            uu[...] = u[f0:f0 + nf]
            vv[...] = v[f0:f0 + nf]

        def write(wnd):
            for t_ in wnd.text.values():
                int(t_[::4096].sum())           # touch one byte per page

        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if len(hs) == 1:
            hs[0].predict_stream(rws[0], f, wid, hgt, 2, read, write, outputs=_lib.OUT_TEXT)
        else:
            _lib.predict_stream_multi(hs, rws, f, wid, hgt, 2, read, write, outputs=_lib.OUT_TEXT)
        return time.perf_counter() - t0

    def ctus(wid, hgt, f):
        return f * (hgt // 64) * (wid // 64) / 4 * len(QPS)

    out = {"frames": args.frames, "steps": args.steps, "qps": list(QPS), "bitdepth": 10, "write": "touch one byte per page",
           "speedup": {}}
    bases = {}
    for wid, hgt in ((1920, 1080), (3840, 2160)):
        key = "%dx%d" % (wid, hgt)
        base = bases[key] = natural(wid, hgt, args.frames, seed=200 + wid)
        for kind in ("static", "letterbox", "mixed", "natural"):
            seq = sequence(kind, base)
            twin = perturbed(*seq)
            legs = {"seq": seq, "twin": twin}
            stream([h], [rows], seq, wid, hgt)          # warm-up of this shape
            times = {k: [] for k in legs}
            frac = {}
            for _ in range(args.steps):
                for k, s in legs.items():
                    h.block_stats(reset=True)
                    times[k].append(stream([h], [rows], s, wid, hgt))
                    b, c = h.block_stats()
                    frac[k] = (c, b)
            assert frac["twin"][0] == frac["twin"][1], (key, kind, frac["twin"])
            best = {k: min(t) for k, t in times.items()}
            out["speedup"]["%s_%s" % (key, kind)] = {
                "ctu_per_s": round(ctus(wid, hgt, args.frames) / best["seq"], 1),
                "twin_ctu_per_s": round(ctus(wid, hgt, args.frames) / best["twin"], 1),
                "computed": frac["seq"][0], "blocks": frac["seq"][1],
                "computed_fraction": round(frac["seq"][0] / frac["seq"][1], 4),
                "ratio": round(best["twin"] / best["seq"], 3),
                "seconds": {k: [round(x, 4) for x in t] for k, t in times.items()}}
            print(kind, key, out["speedup"]["%s_%s" % (key, kind)], file=sys.stderr, flush=True)

    # grouping share: one default window of the 4K natural sequence
    wid, hgt = 3840, 2160
    y, u, v = bases["%dx%d" % (wid, hgt)]
    bpf = (hgt // 64) * (wid // 64)
    wf = max(1, 4800 // bpf)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a[:wf]).view(np.int16)).cuda()   # noqa: E731
    lb, cb = ops.cut_blocks(cuda(y), cuda(u), cuda(v), handle=h)
    rep = torch.empty(wf * bpf, dtype=torch.int32, device="cuda")
    group_ms = {}
    for comp, blk in zip(COMPS, (lb, cb)):
        n = blk.shape[0]
        call = lambda: _lib.check(_lib.lib().pmp_debug_block_groups(      # noqa: E731
            h.ptr, ctypes.c_void_p(blk.data_ptr()), n, blk[0].numel(), 64, ctypes.c_void_p(rep.data_ptr()), None, None))
        call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        e1.synchronize()
        group_ms[comp] = round(e0.elapsed_time(e1) / reps, 4)
    nat = out["speedup"]["%dx%d_natural" % (wid, hgt)]
    nwin = -(-args.frames // wf)
    win_ms = min(nat["seconds"]["seq"]) * 1e3 / nwin
    out["grouping"] = {"window_frames": wf, "blocks": wf * bpf, "ms_per_component": group_ms,
                       "window_ms": round(win_ms, 3),
                       "share_of_window": round(sum(group_ms.values()) / win_ms, 6),
                       "note": "pmp_debug_block_groups (includes its host synchronisation) over the window time of stream_1h"}

    if "parent" in libs:
        builds = {}
        for which in ("this", "parent"):
            use(which)
            hs = [handle() for _ in range(2)]
            builds[which] = hs
        seq = bases["%dx%d" % (wid, hgt)]
        legs = {"stream_1h": lambda hs: stream([hs[0][0]], [hs[0][1]], seq, wid, hgt),
                "multi_2h_dev0": lambda hs: stream([x[0] for x in hs], [x[1] for x in hs], seq, wid, hgt)}
        times = {}
        for which in ("this", "parent"):            # warm-up
            use(which)
            for leg, fn in legs.items():
                fn(builds[which])
        for _ in range(args.steps):
            for leg, fn in legs.items():
                for which in ("parent", "this"):
                    use(which)
                    times.setdefault((which, leg), []).append(fn(builds[which]))
        use("this")
        st = builds["this"][0][0].block_stats()
        ov = {"blocks": st[0], "computed": st[1]}
        for leg in legs:
            for which in ("parent", "this"):
                t = times[(which, leg)]
                ov["%s_%s" % (leg, which)] = {"ctu_per_s": round(ctus(wid, hgt, args.frames) / min(t), 1),
                                              "seconds": [round(x, 4) for x in t],
                                              "spread_pct": round(100 * (max(t) - min(t)) / min(t), 2)}
            ov["%s_this_over_parent" % leg] = round(min(times[("parent", leg)]) / min(times[("this", leg)]), 4)
        out["overhead_%dx%d_natural" % (wid, hgt)] = ov
        for which in ("this", "parent"):
            use(which)
            for x in builds[which]:
                x[0].close()
        use("this")
    h.close()
    return out


if __name__ == "__main__":
    main()
