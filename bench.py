#!/usr/bin/env python
"""Benchmark of the partition-map prediction hot path (BASELINE.json metric: CTUs/sec & 4K frames/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|torch-cuda] [--engine tc|simt]
                    [--workload 1080p10|4k30]

Workload (BASELINE.json configs[1]): a synthetic 1920x1080 10-bit 4:2:0 10-frame sequence (480 64x64 blocks =
120 CTUs per frame), luma + chroma QT+MTT nets at QP 22/27/32/37, QT post-process, map-to-partition decode and frame
assembly.  One "step" = one pass of the whole path over that sequence: 10 frames x 120 CTUs x 4 QPs = 4800 CTU-QP
units (a unit = one 128x128 CTU through luma Q+MSBD, chroma Q+MSBD and both decodes for one QP = 37.164 GFLOP).
N > 1: every rank runs its own sequence (frame sharding, no data-path collective) -> weak scaling.

`value`  : units/s with the frames already resident in HBM (device timing, CUDA events, max over ranks).
`e2e`    : the same through the public API (PartitionPredictor.predict_frames) from pinned HOST frames, H2D of the
           frames and D2H of the int8 partition vectors inside the timed region.
`roofline`: the conv kernel class that dominates the step, algorithmic FLOPs / CUDA-event time of its launches over a
           second pass of the same K steps (per-launch event pairs; `value` is timed without them), against the
           measured bf16 peak, see peaks().
`cpu_baseline`: the oracle port of the reference's CPU path (PyTorch CPU fp32 nets + NumPy post-process/decode),
           timed on this host on a bounded sample of the same workload (rank 0, N=1 only).
`gpu_baseline`: the only GPU implementation the reference has -- its PyTorch modules under torch/cuDNN
           (Inference_QBD.py:223-226) -- as the oracle's plain-torch forwards on cuda:0, fp32 with TF32 off (parity-grade)
           and TF32 on (labelled non-parity), nets only (decode excluded: favours the baseline).
`text_write`: PartitionMat text formatting on the GPU + device->host copy + file write of the step's results
           (Map2Partition.py:400-412), reported separately from `e2e` as SURVEY 8(d) asks.
`decode_report`: count of blocks whose argmin was a float32 near-tie / whose maps hold a value within tolerance of a
           decision threshold (north star: "a reported count of CTUs ...").
`--impl reference`: times that CPU path alone (same metric/config), see reference_main().
`--impl torch-cuda`: times the torch/cuDNN arm alone (same metric/config).
`--workload 4k30`: BASELINE configs[2] -- ONE synthetic 3840x2160 30-frame sequence strong-scaled over the N ranks by
           frame sharding (Map2Partition.py:389-412 makes the gather a concatenation), see fourk_main().
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step returned (the int8 PartitionMat
           vectors of every component and QP) as DIR/<comp>_QP<qp>.npy, see dump_outputs().  The inputs are seeded, so two
           builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WIDTH, HEIGHT, FRAMES = 1920, 1080, 10
QPS = (22, 27, 32, 37)
COMPS = ("Luma", "Chroma")
METRIC = "CTUs/sec (128x128 CTU, luma+chroma QT+MTT nets + post-process + Map2Partition decode, per QP)"
UNIT = "CTU/s"


def workload_config(engine=None):
    """The workload both arms carry (identical dicts: the engine is a top-level key of the line, not part of the workload)."""
    bh, bw = HEIGHT // 64, WIDTH // 64
    return {"workload": "synthetic 1920x1080 10-bit 4:2:0, %d frames, Luma+Chroma x QP 22/27/32/37 (BASELINE configs[1])" % FRAMES,
            "blocks_per_frame": bh * bw, "ctus_per_frame": bh * bw // 4, "frames": FRAMES, "qps": list(QPS),
            "units_per_step": FRAMES * bh * bw * len(QPS) // 4,
            "l2": "no flush: per-step working set (activation arena, GBs) >> 126 MB L2",
            "weights": "Q nets: reference trained .pkl; MSBD nets: seeded random (trained *_BD_*.pkl absent offline)"}


def peaks():
    """Roofline denominators: the B200 peaks measured for this project (BASELINE.md section 2), unless a
    MEASURED_PEAKS.json beside this file holds peaks measured on the card at hand."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"],
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6446.6, "bf16_burst": 1660.1, "bf16_sustained": 1413.7,
            "src": "measured on a B200, power limit not recorded (BASELINE.md section 2)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons, pw = [], [], set(), []
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def load_predictor(dev, engine, chunk):
    from pmp_vvc_tip2023_b200.pipeline import PartitionPredictor
    pp = PartitionPredictor(dev, engine=engine, chunk=chunk)
    pp.load_pkls(os.path.join(ROOT, "trained_models"), missing_bd="seeded")
    return pp


def make_frames(seed, width=WIDTH, height=HEIGHT, frames=FRAMES):
    from pmp_vvc_tip2023_b200 import synth
    # one synthetic frame generator call per distinct frame is slow in numpy at 1080p: build 2 and alternate with shifts
    y, u, v = synth.synth_yuv420(width, height, 2, seed=seed)
    idx = [i % 2 for i in range(frames)]
    ys = np.stack([np.roll(y[k], 8 * i, axis=1) for i, k in enumerate(idx)])
    us = np.stack([np.roll(u[k], 4 * i, axis=1) for i, k in enumerate(idx)])
    vs = np.stack([np.roll(v[k], 4 * i, axis=1) for i, k in enumerate(idx)])
    return ys, us, vs


# values kept per output by dump_outputs: 8 outputs x 2^20 float32 = 32 MB per dump (a step returns 51.6 M int8 values)
DUMP_SAMPLE = 1 << 20


def dump_outputs(out_dir, results, sample=DUMP_SAMPLE):
    """Write {(comp, qp): int8 tensor [F, per-frame values]} as out_dir/<comp>_QP<qp>.npy, float32, flattened.  An output
    longer than `sample` is reduced to the values at `sample` sorted positions drawn with a fixed seed (the same positions
    for every output of that length, in every run).  Returns {name: number of values written}."""
    os.makedirs(out_dir, exist_ok=True)
    written = {}
    for (comp, qp), vals in sorted(results.items()):
        a = vals.cpu().numpy().reshape(-1)
        if a.size > sample:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, size=sample, replace=False))]
        name = "%s_QP%d" % (comp, qp)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))
        written[name] = int(a.size)
    return written


def kernel_source_sha():
    """sha256 over the CUDA sources: ties a committed ncu traffic summary to the kernels it was measured on."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pmp_vvc_tip2023_b200", "csrc")
    for f in sorted(os.listdir(d)):
        h.update(f.encode())
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(blocks_per_launch):
    """(bytes per conv_tc launch, provenance) from the newest committed ncu DRAM summary, or (None, why) when that file
    was measured on other kernel sources than the ones loaded now (a stale constant is worse than none)."""
    import glob
    cands = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    if not cands:
        return None, "no profiles/r*_traffic.json"
    tj = json.load(open(cands[-1]))
    name = os.path.basename(cands[-1])
    if tj.get("kernel_source_sha") != kernel_source_sha():
        return None, "%s was measured on kernel sources %s, loaded sources are %s: not reported" % (
            name, tj.get("kernel_source_sha"), kernel_source_sha())
    return tj["conv_tc_dram_bytes_per_launch_per_block"] * blocks_per_launch, \
        "%s (%s); per launch and block, scaled to %d blocks per launch" % (name, tj["source"], blocks_per_launch)


# ------------------------------------------------------------------------------------------------------
# torch/cuDNN arm: the reference's own GPU implementation (stock PyTorch modules, Inference_QBD.py:223-226)
# ------------------------------------------------------------------------------------------------------
def torch_cuda_sample(dev, nblocks=480, reps=3):
    """oracle.nets_ref (the reference's forwards in plain torch) on the GPU: one 1080p frame, luma + chroma, QP 32.
    Returns {tf32 off / on: CTU/s}; nets only."""
    from oracle import nets_ref
    cp = CpuPath()
    by, bu, bv = (b[:nblocks] for b in cp.blocks)
    d = torch.device("cuda", dev)
    xs = {"Luma": torch.from_numpy(by.astype(np.float32)).unsqueeze(1).to(d), "Chroma": nets_ref.chroma_net_input(by, bu, bv).to(d)}
    sds = {c: tuple({k: t.to(d) for k, t in sd.items()} for sd in cp.sd[c]) for c in COMPS}
    out = {}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        for tf32 in (False, True):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            run = lambda: [nets_ref.predict_maps(sds[c][0], sds[c][1], xs[c], c == "Luma", batch=240) for c in COMPS]
            run(); run()
            torch.cuda.synchronize(d)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                res = run()
            e1.record()
            torch.cuda.synchronize(d)
            out["tf32" if tf32 else "fp32"] = (nblocks / 4.0) * reps / (e0.elapsed_time(e1) * 1e-3)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    return {"value": out["fp32"], "unit": UNIT, "kind": "torch-cuda (oracle.nets_ref = the reference's forwards, cuDNN fp32, TF32 off)",
            "tf32_value": out["tf32"], "tf32_note": "TF32 on: NOT parity-grade (SURVEY 7.3: TF32 operands miss the 1e-2 bar)",
            "sample": "%d blocks (one 1080p frame), luma+chroma Q+MSBD nets, QP 32, batch 240, %d reps, cudnn.benchmark; "
                      "post-process/decode excluded (favours this baseline)" % (nblocks, reps),
            "torch": torch.__version__, "cudnn": torch.backends.cudnn.version()}


def torch_cuda_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    if not torch.cuda.is_available():
        raise SystemExit("--impl torch-cuda needs a CUDA device")
    g = torch_cuda_sample(0, reps=max(args.steps, 1))
    out = {"impl": "torch-cuda", "metric": METRIC, "value": g["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic", "config": workload_config(), "engine": "torch-cudnn", "gpu_baseline": g}
    print(json.dumps(out))
    return 0


def text_write_leg(pp, results, frames, out_dir=None):
    """Format the step's int8 vectors as PartitionMat text on the GPU, copy to the host and write the files
    (Map2Partition.py:400-412).  Returns timings; files go to a temp dir and are removed unless out_dir is given."""
    import shutil
    from pmp_vvc_tip2023_b200 import ops
    tmp = out_dir or tempfile.mkdtemp(prefix="pmp_text_")
    os.makedirs(tmp, exist_ok=True)
    torch.cuda.synchronize()
    t_fmt = t_d2h = t_wr = 0.0
    nbytes = 0
    for (comp, qp), vals in results.items():
        t0 = time.perf_counter()
        text = ops.format_text(vals, handle=pp.handle)          # synchronises (returns the byte count)
        t1 = time.perf_counter()
        host = text.cpu().numpy()
        t2 = time.perf_counter()
        with open(pp.partition_path(tmp, "bench_seq", comp, qp), "wb") as fp:
            fp.write(host.tobytes())
        t3 = time.perf_counter()
        t_fmt += t1 - t0; t_d2h += t2 - t1; t_wr += t3 - t2
        nbytes += host.size
    if not out_dir:
        shutil.rmtree(tmp, ignore_errors=True)
    return {"format_ms": 1e3 * t_fmt, "d2h_ms": 1e3 * t_d2h, "file_write_ms": 1e3 * t_wr, "text_bytes": int(nbytes),
            "files": len(results), "frames": frames}


# ------------------------------------------------------------------------------------------------------
# CPU path (oracle port of the reference): used for cpu_baseline and --impl reference
# ------------------------------------------------------------------------------------------------------
class CpuPath:
    def __init__(self):
        from oracle import decode_ref, nets_ref, postproc_ref
        from pmp_vvc_tip2023_b200 import synth
        from pmp_vvc_tip2023_b200.weights import load_reference_pkl
        self.nets_ref, self.postproc_ref, self.decode_ref = nets_ref, postproc_ref, decode_ref
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        self.sd = {}
        for comp in COMPS:
            sdq = load_reference_pkl(os.path.join(ROOT, "trained_models", "%s_Q_32.pkl" % comp))
            sdb = {k: torch.from_numpy(v) for k, v in synth.seeded_state_dict(comp + "_MSBD", 1032 + (0 if comp == "Luma" else 500)).items()}
            self.sd[comp] = (sdq, sdb)
        y, u, v = make_frames(0)
        self.blocks = nets_ref.cut_blocks(y[:1], u[:1], v[:1], True)      # 480 blocks of frame 0

    def run(self, nblocks, lo=0):
        """nblocks blocks (luma + chroma, one QP) through nets -> post-process -> NumPy decode.  Returns (s_nets, s_post)."""
        by, bu, bv = (b[lo:lo + nblocks] for b in self.blocks)
        t_net = t_post = 0.0
        for comp in COMPS:
            luma = comp == "Luma"
            t0 = time.perf_counter()
            x = torch.from_numpy(by.astype(np.float32)).unsqueeze(1) if luma else self.nets_ref.chroma_net_input(by, bu, bv)
            qt, bt, dire = self.nets_ref.predict_maps(self.sd[comp][0], self.sd[comp][1], x, luma, batch=200)
            t1 = time.perf_counter()
            qi = self.postproc_ref.eli_structural_error(qt.numpy())[:, 0]
            btn, din = bt.numpy(), dire.numpy()
            for b in range(qi.shape[0]):       # single Python thread, as Map2Partition.py:389-399 runs it
                self.decode_ref.map_to_partition(qi[b], btn[b], din[b], 1 if luma else 2)
            t2 = time.perf_counter()
            t_net += t1 - t0
            t_post += t2 - t1
        return t_net, t_post


def cpu_baseline_sample(budget_s=20.0):
    cp = CpuPath()
    tn, tp = cp.run(8)                                     # calibrate
    per_block = (tn + tp) / 8
    n = int(max(8, min(480, budget_s / max(per_block, 1e-6))))
    tn, tp = cp.run(n)
    return {"value": (n / 4.0) / (tn + tp), "unit": UNIT, "cores": cp.cores, "kind": "port",
            "sample": "%d blocks (=%g CTUs) of frame 0, luma+chroma, QP 32: torch-CPU fp32 nets (%d threads, batch 200) "
                      "%.2f s + NumPy post-process/decode (1 thread, as the reference runs it) %.2f s" % (n, n / 4.0, cp.cores, tn, tp),
            "nets_s": tn, "post_s": tp}


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cp = CpuPath()
    tn, tp = cp.run(8)
    per_block = (tn + tp) / 8
    total_budget = 150.0
    n = int(max(4, min(480, total_budget / max(args.steps + args.warmup, 1) / max(per_block, 1e-6))))
    for _ in range(args.warmup):
        cp.run(n)
    t0 = time.perf_counter()
    tn = tp = 0.0
    for _ in range(args.steps):
        a, b = cp.run(n)
        tn += a; tp += b
    el = time.perf_counter() - t0
    value = args.steps * (n / 4.0) / el
    sample = ("%d blocks (=%g CTUs) per step of frame 0, luma+chroma, QP 32; nets %.2f s (torch CPU fp32, %d threads), "
              "post-process+decode %.2f s (NumPy, 1 thread)" % (n, n / 4.0, tn, cp.cores, tp))
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * el / max(args.steps, 1), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(), "engine": "reference-cpu",
           "units_timed_per_step": n / 4.0,
           "extrapolation": "each step times a bounded sample (%d blocks of frame 0, QP 32) of the workload in `config` and the "
                            "rate is quoted per CTU: units_per_step in `config` is the nominal workload, not what a step ran" % n,
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cp.cores, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "note": "reference is Python/PyTorch (not installable as a binary): its CPU path is the oracle port, "
                   "pinned to the reference's own outputs by tests/golden"}
    print(json.dumps(out))
    return 0


# ------------------------------------------------------------------------------------------------------
# BASELINE configs[2]: ONE 3840x2160 x 30-frame sequence, frames sharded over the N ranks (strong scaling)
# ------------------------------------------------------------------------------------------------------
def fourk_main(args):
    """Each rank predicts a contiguous frame range of the same sequence with the product path (PartitionPredictor, the
    engine behind Inference_QBD --gpus N), formats its PartitionMat text segments on the GPU, and rank 0 gathers them
    (NCCL gather of the uint8 text over NVLink, one device->host copy) and concatenates in frame order -- exactly the file
    layout (Map2Partition.py:389-412).  `value`: device-resident frames -> int8 vectors; `e2e`: pinned host frames ->
    rank 0 holds every file's bytes in host memory (gather included); file write reported separately."""
    import hashlib
    import torch.distributed as dist
    from pmp_vvc_tip2023_b200 import ops
    W4, H4, F4 = 3840, 2160, 30
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pp = load_predictor(local, args.engine, args.chunk)
    y, u, v = make_frames(400, W4, H4, F4)                     # every rank builds the same sequence, keeps what it needs
    # Shards: the F4 x 4 (QP, frame) pairs in QP-major order, split evenly over the ranks -- rank r predicts, for one or two
    # QPs, a contiguous frame range of both components.  (Sharding whole frames with all four QPs leaves 30 frames on 8
    # GPUs at 4 vs 3.75 frames per rank, a 93.75 % ceiling; 120 pairs split 15 / 15 / ... exactly.)  Every file is still a
    # concatenation of rank-ordered segments.  --shard frames selects the plain frame ranges.
    from pmp_vvc_tip2023_b200 import sharding

    def shard_of(r):                                           # [(qp, frame_lo, frame_hi)] of rank r
        fn = sharding.frame_shards if args.shard == "frames" else sharding.qp_frame_shards
        return [(QPS[qi], a, b) for qi, a, b in fn(F4, len(QPS), world, r)]
    pieces = shard_of(rank)
    f_lo = min([p_[1] for p_ in pieces], default=0)
    f_hi = max([p_[2] for p_ in pieces], default=0)
    hy, hu, hv = (torch.from_numpy(np.ascontiguousarray(a[f_lo:f_hi]).view(np.int16)).pin_memory() for a in (y, u, v))
    dy, du, dv = (t.cuda() for t in (hy, hu, hv))
    bh, bw = H4 // 64, W4 // 64
    units = F4 * bh * bw * len(QPS) / 4.0
    keys = [(c, q) for c in COMPS for q in QPS]
    # consecutive pieces with the same frame range share one predict_frames call (one block cut for all their QPs)
    calls = sharding.group_calls(pieces)
    h2d_bytes = sum(2 * (b - a) * (W4 * H4 * 3 // 2) for _, a, b in calls)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def predict(ty, tu, tv):
        res = {}
        for qs, a, b in calls:
            res.update(pp.predict_frames(ty[a - f_lo:b - f_lo], tu[a - f_lo:b - f_lo], tv[a - f_lo:b - f_lo], qps=tuple(qs)))
        return res

    def step_device():
        return predict(dy, du, dv)

    gathered = {}

    def step_e2e():
        res = predict(hy, hu, hv)
        texts = {k: (ops.format_text(res[k], handle=pp.handle) if k in res else torch.empty(0, dtype=torch.uint8, device="cuda")) for k in keys}
        if world == 1:
            for k in keys:
                gathered[k] = pp.to_host_pinned(("text",) + k, texts[k], sync=False)     # reusable pinned staging
            torch.cuda.synchronize()
            return
        sizes = torch.tensor([texts[k].numel() for k in keys], dtype=torch.int64, device="cuda")
        all_sizes = [torch.empty_like(sizes) for _ in range(world)]
        dist.all_gather(all_sizes, sizes)
        all_sizes = torch.stack(all_sizes).cpu()                # [world, 8]
        for i, k in enumerate(keys):
            mx = int(all_sizes[:, i].max())
            buf = torch.empty(mx, dtype=torch.uint8, device="cuda")
            buf[:texts[k].numel()] = texts[k]
            outs = [torch.empty(mx, dtype=torch.uint8, device="cuda") for _ in range(world)] if rank == 0 else None
            dist.gather(buf, outs, dst=0)                       # NCCL over NVLink
            if rank == 0:
                gathered[k] = pp.to_host_pinned(("text",) + k, torch.cat([outs[r][:int(all_sizes[r, i])] for r in range(world)]),
                                                sync=False)
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(args.warmup, 1)):
        step_device()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = pp.handle.launch_count()
    ms = timed(step_device, args.steps)
    launches = pp.handle.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    counts = pp.counts()["total"]
    cnt = torch.tensor([counts["blocks"], counts["near_tie_blocks"], counts["near_threshold_blocks"], counts["fp16_saturation_events"],
                        counts["near_threshold_blocks_tight"], h2d_bytes],
                       dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(cnt)
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0
    sha = {"%s_QP%d" % k: hashlib.sha256(gathered[k].numpy().tobytes()).hexdigest()[:16] for k in keys}
    tmp = args.out_dir or tempfile.mkdtemp(prefix="pmp_4k30_")
    os.makedirs(tmp, exist_ok=True)
    t0 = time.perf_counter()
    nbytes = 0
    for k in keys:
        with open(pp.partition_path(tmp, "synth4k_3840x2160_30", k[0], k[1]), "wb") as fp:
            fp.write(gathered[k].numpy().tobytes())
        nbytes += gathered[k].numel()
    t_write = time.perf_counter() - t0
    if not args.out_dir:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
    verified = None
    if args.verify and world > 1:
        # rank 0 alone over the whole sequence: the concatenation of the shards must be the same bytes
        fy, fu, fv = (torch.from_numpy(a.view(np.int16)).cuda() for a in (y, u, v))
        full = pp.predict_frames(fy, fu, fv, qps=QPS)
        verified = all(torch.equal(ops.format_text(full[k], handle=pp.handle).cpu(), gathered[k]) for k in keys)
        assert verified, "sharded PartitionMat bytes differ from the single-GPU result"
    value = units * args.steps / (ms * 1e-3)
    e2e_value = units * args.steps / (ms_e2e * 1e-3)
    cfg = {"workload": "synthetic 3840x2160 10-bit 4:2:0, 30 frames, ONE sequence, Luma+Chroma x QP 22/27/32/37, %s sharded "
                       "over %d GPU(s) (BASELINE configs[2])" % ("(QP, frame) pairs" if args.shard == "frame-qp" else "frames", world),
           "blocks_per_frame": bh * bw, "frames": F4, "qps": list(QPS), "units_per_step": units, "engine": args.engine,
           "shard": args.shard, "qp_frame_ranges_per_rank": [shard_of(r) for r in range(world)],
           "l2": "no flush: per-step working set >> 126 MB L2",
           "weights": "Q nets: reference trained .pkl; MSBD nets: seeded random (trained *_BD_*.pkl absent offline)"}
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f16x3(split)+f32acc", "data": "synthetic", "config": cfg,
           "frames_4k_per_s_all_qps": F4 * args.steps / (ms * 1e-3), "frame_qps_4k_per_s": F4 * len(QPS) * args.steps / (ms * 1e-3),
           "gpu_launches": int(launches), "clocks": clocks,
           "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                   "h2d_bytes_per_step": int(cnt[5]), "d2h_bytes_per_step": int(nbytes),
                   "note": "pinned host frames -> predict -> GPU text formatting -> NCCL gather to rank 0 -> host bytes of the 8 "
                           "PartitionMat files"},
           "file_write": {"ms": 1e3 * t_write, "bytes": int(nbytes), "e2e_plus_write_ctu_per_s": units / (ms_e2e * 1e-3 / args.steps + t_write)},
           "text_sha256_16": sha, "verified_equal_to_single_gpu": verified,
           "decode_report": {"near_tol": 1e-2, "block_qps": int(cnt[0]), "near_tie_blocks": int(cnt[1]),
                             "near_threshold_blocks": int(cnt[2]), "near_threshold_blocks_tight_1e-4": int(cnt[4]),
                             "fp16_saturation_events": int(cnt[3])}}
    print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="b200", choices=["b200", "reference", "torch-cuda"])
    ap.add_argument("--workload", type=str, default="1080p10", choices=["1080p10", "4k30"])
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-text-write", action="store_true")
    ap.add_argument("--verify", action="store_true", help="4k30: rank 0 recomputes the whole sequence alone and compares bytes")
    ap.add_argument("--shard", type=str, default="frame-qp", choices=["frame-qp", "frames"],
                    help="4k30: shard (QP, frame) pairs evenly over the ranks (default) or whole frame ranges with all QPs")
    ap.add_argument("--out-dir", type=str, default=None, help="4k30 / text_write: where PartitionMat files are written (default: a temp dir)")
    ap.add_argument("--engine", type=str, default="tc", choices=["tc", "simt"])
    ap.add_argument("--chunk", type=int, default=4800)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write what the last timed step computed as DIR/<comp>_QP<qp>.npy (float32, a fixed seeded "
                         "sample of %d values per output)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "1080p10"):
        ap.error("--dump-outputs is implemented for --impl b200 --workload 1080p10")
    if args.impl == "reference":
        return reference_main(args)
    if args.impl == "torch-cuda":
        return torch_cuda_main(args)
    if args.workload == "4k30":
        return fourk_main(args)
    args.warmup = max(args.warmup, 3)

    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from pmp_vvc_tip2023_b200 import netspec
    pp = load_predictor(local, args.engine, args.chunk)
    h = pp.handle
    y, u, v = make_frames(100 + rank)
    hy, hu, hv = (torch.from_numpy(a.view(np.int16)).pin_memory() for a in (y, u, v))
    dy, du, dv = (t.cuda() for t in (hy, hu, hv))
    bh, bw = HEIGHT // 64, WIDTH // 64
    units = FRAMES * bh * bw * len(QPS) / 4.0
    per = 2 * (bh * 16) * (bw * 16) + (bh * 8) * (bw * 8) + 3 * (bh * 16) * (bw * 16)
    host_out = {(c, q): torch.empty((FRAMES, per), dtype=torch.int8).pin_memory() for c in COMPS for q in QPS}

    def step_device():
        return pp.predict_frames(dy, du, dv, qps=QPS)

    def step_e2e():
        pp.predict_frames(hy, hu, hv, qps=QPS, host_out=host_out)      # D2H of each component overlaps the next one
        pp.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(ms of `steps` calls of fn, what the last call returned)"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = h.launch_count()
    ms, last = timed(step_device, args.steps)           # `value`: no per-launch events in the stream
    launches = h.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    dumped = dump_outputs(args.dump_outputs, last) if args.dump_outputs and rank == 0 else None
    del last
    # roofline pass: the same K steps again with a CUDA-event pair around every launch (the events sit between the
    # kernels, which switches off the programmatic-dependent-launch overlap, hence a separate pass)
    prof, ms_prof = {}, None
    if not args.no_profile:
        h.profile(2)
        ms_prof, _ = timed(step_device, args.steps)
        prof = h.profile_read()
        h.profile(0)

    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    decode_report = pp.counts() if rank == 0 else None
    text_leg = None
    if rank == 0 and not args.no_text_write:
        text_leg = text_write_leg(pp, step_device(), FRAMES, args.out_dir)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    pk = peaks()
    value = world * units * args.steps / (ms * 1e-3)
    e2e_value = world * units * args.steps / (ms_e2e * 1e-3)
    dom = "conv_tc" if args.engine == "tc" and prof.get("conv_tc", {}).get("ms", 0) > 0 else "conv_simt"
    roof = None
    if not args.no_profile and prof.get(dom, {}).get("ms", 0) > 0:
        p = prof[dom]
        ach = p["flops"] / (p["ms"] * 1e-3) / 1e12
        blocks_per_launch = min(args.chunk, FRAMES * (HEIGHT // 64) * (WIDTH // 64))
        traffic, traffic_src = measured_traffic(blocks_per_launch) if dom == "conv_tc" else (None, "not measured for this engine")
        roof = {"kernel": dom, "bound": "tensor", "achieved": ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["bf16_sustained"], "traffic": traffic, "traffic_src": traffic_src,
                "peak_src": pk["src"] + ", sustained bf16 (kernel timed inside a long step)",
                "launches": p["launches"], "avg_launch_ms": p["ms"] / max(p["launches"], 1),
                "algorithmic_flops_per_launch": p["flops"] / max(p["launches"], 1),
                # every operand tensor of the launch once at 4 B/element (hi + lo planes); counted by the library per launch
                "algorithmic_hbm_bytes_per_launch": p["bytes"] / max(p["launches"], 1),
                "algorithmic_hbm_gbs": p["bytes"] / (p["ms"] * 1e-3) / 1e9 if p["ms"] > 0 else None,
                "kernel_source_sha": kernel_source_sha(),
                "share_of_step": p["ms"] / ms_prof, "profiled_pass_ms_per_step": ms_prof / args.steps,
                "note": "algorithmic FLOPs = 2*MACs of the fp32 reference convs; the TC engine issues 3 fp16 MMA passes per "
                        "MAC (split precision), so issued tensor work = 3x this"}
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f16x3(split)+f32acc" if args.engine == "tc" else "f32", "data": "synthetic",
           "config": workload_config(), "engine": args.engine,
           "frames_per_s_1080p_all_qps": world * FRAMES * args.steps / (ms * 1e-3),
           "frame_qp_per_s_4k_equiv": value / 495.0,
           "algorithmic_tflops": value * netspec.FLOPS_PER_CTU / 1e12,
           "gpu_launches": int(launches), "clocks": clocks,
           "e2e": {"value": e2e_value, "unit": UNIT,
                   "h2d_bytes_per_step": int(hy.numel() * 2 + hu.numel() * 2 + hv.numel() * 2),
                   "d2h_bytes_per_step": int(sum(t.numel() for t in host_out.values())),
                   "ms_per_step": ms_e2e / args.steps},
           "roofline": roof,
           "kernel_classes_ms_per_step": {k: p["ms"] / args.steps for k, p in prof.items() if p["launches"]},
           # the integer / element-wise kernel classes against the HBM roofline: algorithmic bytes (DESIGN.md section 4.3)
           # over the CUDA-event time of their launches in the profiled pass
           "hbm_kernels": {k: {"achieved_gbs": p["bytes"] / (p["ms"] * 1e-3) / 1e9, "peak_gbs": pk["hbm_gbs"],
                               "frac": p["bytes"] / (p["ms"] * 1e-3) / 1e9 / pk["hbm_gbs"], "launches": p["launches"]}
                           for k, p in prof.items() if p["launches"] and p["bytes"] > 0 and p["ms"] > 0 and not k.startswith("conv")}}
    tot = decode_report["total"]
    out["decode_report"] = {"near_tol": 1e-2, "block_qps": tot["blocks"], "near_tie_blocks": tot["near_tie_blocks"],
                            "near_threshold_blocks": tot["near_threshold_blocks"],
                            "near_tight_tol": 1e-4, "near_threshold_blocks_tight": tot["near_threshold_blocks_tight"],
                            "near_tie_ctus_upper_bound": min(tot["near_tie_blocks"], tot["blocks"] // 4),
                            "fp16_saturation_events": tot["fp16_saturation_events"],
                            "note": "per 64x64 block and QP over the last step (a 128x128 CTU = 4 blocks): near_tie = the "
                                    "argmin's runner-up lies within the reference's float32 evaluation noise (flags bit 0); "
                                    "near_threshold = a map value within near_tol of a rounding threshold (bits 1-3; with ~1,600 map values per block "
                                    "nearly every block has one at 1e-2, hence the second count at near_tight_tol = 2x the "
                                    "largest measured map error, bits 4-6). Only "
                                    "these blocks may legitimately differ from a float32 evaluation of the reference."}
    if text_leg:
        sec = (text_leg["format_ms"] + text_leg["d2h_ms"] + text_leg["file_write_ms"]) * 1e-3
        text_leg["ctu_per_s_text_only"] = units / sec
        text_leg["ctu_per_s_e2e_plus_text"] = units / (ms_e2e * 1e-3 / args.steps + sec)
        out["text_write"] = text_leg
    if dumped:
        out["dump_outputs"] = {"dir": args.dump_outputs, "values": dumped, "dtype": "float32",
                               "sample": "int8 PartitionMat vectors of the last timed step, flattened; outputs longer than "
                                         "%d values sampled at fixed seeded positions" % DUMP_SAMPLE}
    if world == 1 and not args.no_gpu_baseline:
        pp.close()
        torch.cuda.empty_cache()
        out["gpu_baseline"] = torch_cuda_sample(local)
        out["gpu_baseline"]["e2e_over_gpu_baseline"] = e2e_value / out["gpu_baseline"]["value"]
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_sample()
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
