"""Exact reuse of repeated blocks in the window pipeline: the grouping (pmp_debug_block_groups) against a numpy "lowest
equal index" reference, with forced fingerprint collisions; the outputs of pmp_predict_host, pmp_predict_stream,
pmp_predict_stream_multi and pmp_predict_stream_ex on content with repeats against PartitionPredictor (the csrc/ path,
which computes every block); the work counted by pmp_block_stats and the profile; the saturation stop; the native tool's
"Block reuse:" line; and handles on distinct devices."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from pmp_vvc_tip2023_b200 import _lib, Inference_QBD, ops, synth
from pmp_vvc_tip2023_b200.netspec import QPS
from pmp_vvc_tip2023_b200.pipeline import PartitionPredictor
from tests import cases
from tests.test_gpu_stream import (COMPS, MODELS, Collector, _report_line, _saturating_luma_q, _write_yuv,  # noqa: F401
                                   exported, native_tool)

pytestmark = pytest.mark.gpu
BLOCK_BYTES = (68 * 68, 3 * 34 * 34)
SWEEP = [ops.DEFAULT_LAMB, cases.LAMB_SETS["a"], cases.LAMB_SETS["b"], cases.LAMB_SETS["c"]]
REPORT_KEYS = ("blocks", "near_tie_blocks", "near_threshold_blocks", "near_threshold_blocks_tight")


# ---- content with repeats -----------------------------------------------------------------------------------------------
def content(kind, width, height, frames, bitdepth, seed):
    """y [F,H,W], u/v [F,H/2,W/2] of one kind, seeded from synth.synth_yuv420."""
    y, u, v = synth.synth_yuv420(width, height, frames, seed=seed, bitdepth=bitdepth)
    top = 1023 if bitdepth == 10 else 255
    if kind == "natural":
        return y, u, v
    if kind == "static":                # frame 0 repeated
        return tuple(np.repeat(a[:1], frames, 0) for a in (y, u, v))
    if kind == "letterbox":             # black bars of 140 rows at 1080p; below, 72 rows: a whole block row
        bar = max(72, 2 * round(70 * height / 1080))
        black_y, black_c = (64, 512) if bitdepth == 10 else (16, 128)
        y[:, :bar], y[:, height - bar:] = black_y, black_y
        for c in (u, v):
            c[:, :bar // 2], c[:, (height - bar) // 2:] = black_c, black_c
        return y, u, v
    if kind == "flat":                  # one constant per frame and plane
        rng = np.random.default_rng([seed, 7])
        for a in (y, u, v):
            a[:] = rng.integers(0, top + 1, size=(frames, 1, 1)).astype(a.dtype)
        return y, u, v
    if kind == "tiled":                 # frame f: one 64x64 luma tile with its 32x32 chroma, repeated
        ty, tu, tv = y[:, 64:128, 64:128], u[:, 32:64, 32:64], v[:, 32:64, 32:64]
        reps = (1, -(-height // 64), -(-width // 64))
        return (np.ascontiguousarray(np.tile(ty, reps)[:, :height, :width]),
                np.ascontiguousarray(np.tile(tu, reps)[:, :height // 2, :width // 2]),
                np.ascontiguousarray(np.tile(tv, reps)[:, :height // 2, :width // 2]))
    if kind == "alias":                 # frame f+1 = frame f + 1 on samples = 0 (mod 4) below 1023: the same cut blocks
        assert bitdepth == 10
        for a in (y, u, v):
            for f in range(1, frames):
                p = a[f - 1]
                a[f] = p + ((p % 4 == 0) & (p < 1023)).astype(a.dtype)
        return y, u, v
    if kind == "mixed":                 # natural frames interleaved with repeats
        idx = [0, 0, 1, 2, 2, 0, 3, 3, 1, 4][:frames]
        idx += list(range(frames - len(idx)))
        return tuple(np.ascontiguousarray(a[idx]) for a in (y, u, v))
    raise KeyError(kind)


def perturbed(y, u, v):
    """A twin of the same shape whose blocks all differ: per (frame, block) a mark in two luma samples of the block and
    in one U and one V sample of its chroma (the chroma input's pooled luma may not see the luma mark)."""
    y, u, v = y.copy(), u.copy(), v.copy()
    f, hgt, wid = y.shape
    top = 1023 if y.dtype == np.uint16 else 255
    step = 4 if y.dtype == np.uint16 else 1         # one level after the cut's 10 -> 8-bit reduction
    bh, bw = hgt // 64, wid // 64
    for i in range(bh):
        for j in range(bw):
            k = (np.arange(f) * bh + i) * bw + j    # unique per (frame, block) below 65,536 blocks
            lo, hi = (k % 256) * step, (k // 256 % 256) * step
            y[:, 64 * i + 30, 64 * j + 30], y[:, 64 * i + 31, 64 * j + 30] = lo, hi
            u[:, 32 * i + 15, 32 * j + 15], v[:, 32 * i + 15, 32 * j + 15] = lo, hi
    return y, u, v


def _cuda(a):
    return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda()


def distinct_counts(y, u, v, wf):
    """[(N, distinct luma, distinct chroma)] per window of wf frames, from ops.cut_blocks and numpy unique."""
    f, hgt, wid = y.shape
    bpf = (hgt // 64) * (wid // 64)
    lb, cb = ops.cut_blocks(_cuda(y), _cuda(u), _cuda(v))
    blk = [lb.cpu().numpy().reshape(f * bpf, -1), cb.cpu().numpy().reshape(f * bpf, -1)]
    out = []
    for f0 in range(0, f, wf):
        sl = slice(f0 * bpf, min(f, f0 + wf) * bpf)
        out.append((sl.stop - sl.start,) + tuple(len(np.unique(b[sl], axis=0)) for b in blk))
    return out


def expected_stats(counts, passes):
    """(blocks, computed) of `passes` net passes per component and window."""
    return (sum(2 * n for n, _, _ in counts) * passes, sum(dl + dc for _, dl, dc in counts) * passes)


# ---- 1. grouping ---------------------------------------------------------------------------------------------------------
def _block_set(kind, n, block_bytes, seed):
    rng = np.random.default_rng([seed, n, block_bytes])
    by, bu, bv = synth.synth_blocks(min(n, 256), seed=seed)
    base = by.reshape(len(by), -1) if block_bytes == BLOCK_BYTES[0] else np.concatenate(
        [by[:, ::2, ::2][:, :34, :34].reshape(len(by), -1), bu.reshape(len(by), -1), bv.reshape(len(by), -1)], 1)
    if kind == "all_equal":
        return np.repeat(base[:1], n, 0)
    b = base[np.arange(n) % len(base)].copy()
    # every block distinct: its index in two bytes at a position that varies with the block
    pos = rng.integers(0, block_bytes - 1, size=n)
    b[np.arange(n), pos] = (np.arange(n) & 255).astype(np.uint8)
    b[np.arange(n), pos + 1] = (np.arange(n) >> 8).astype(np.uint8)
    b[np.arange(n), 0] ^= (np.arange(n) % 3 == 0).astype(np.uint8)      # and some differ in their first word too
    if kind == "planted":
        dst = rng.choice(n, size=n // 3, replace=False)
        src = rng.integers(0, n, size=n // 3)
        b[dst] = b[src]
        b[rng.integers(0, n, size=n // 10)] = base[0]                   # one value repeated many times
    return np.ascontiguousarray(b)


def lowest_equal_index(b):
    """rep[i] = the lowest j with b[j] == b[i] (numpy reference)."""
    _, first, inverse = np.unique(b, axis=0, return_index=True, return_inverse=True)
    return first[inverse.reshape(-1)]


def debug_groups(h, blocks, hash_bits):
    n, nbytes = blocks.shape
    dev = torch.from_numpy(blocks).cuda()
    rep = torch.full((max(n, 1),), -1, dtype=torch.int32, device="cuda")
    nd = ctypes.c_int(-1)
    _lib.check(_lib.lib().pmp_debug_block_groups(h.ptr, ctypes.c_void_p(dev.data_ptr()), n, nbytes, hash_bits,
                                                 ctypes.c_void_p(rep.data_ptr()), ctypes.byref(nd), None))
    return rep[:n].cpu().numpy(), nd.value


@pytest.fixture(scope="module")
def handle():
    h = _lib.Handle(0)
    yield h
    h.close()


@pytest.mark.parametrize("hash_bits", [64, 4, 0])
@pytest.mark.parametrize("block_bytes", BLOCK_BYTES)
@pytest.mark.parametrize("kind", ["planted", "all_equal", "all_distinct", "one"])
def test_grouping_is_exact(handle, kind, block_bytes, hash_bits):
    n = 1 if kind == "one" else (20000 if hash_bits else 512)
    b = _block_set("all_distinct" if kind == "one" else kind, n, block_bytes, seed=11)
    rep, nd = debug_groups(handle, b, hash_bits)
    want = lowest_equal_index(b)
    assert np.array_equal(rep, want), (kind, block_bytes, hash_bits, np.nonzero(rep != want)[0][:10])
    assert nd == int((want == np.arange(n)).sum())
    if kind == "all_equal":
        assert nd == 1
    if kind in ("all_distinct", "one"):
        assert nd == n


def test_grouping_arguments(handle):
    L = _lib.lib()
    b = torch.zeros(8 * 4624, dtype=torch.uint8, device="cuda")
    rep = torch.zeros(8, dtype=torch.int32, device="cuda")
    nd = ctypes.c_int(-1)
    p, r = ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(rep.data_ptr())
    for args in ((p, -1, 4624, 64, r), (p, 8, 4622, 64, r), (p, 8, 0, 64, r), (p, 8, 4624, 65, r), (p, 8, 4624, -1, r),
                 (None, 8, 4624, 64, r), (p, 8, 4624, 64, None), (ctypes.c_void_p(b.data_ptr() + 2), 8, 4624, 64, r)):
        assert L.pmp_debug_block_groups(handle.ptr, *args, ctypes.byref(nd), None) == -1, args
    assert L.pmp_debug_block_groups(handle.ptr, p, 0, 4624, 64, r, ctypes.byref(nd), None) == 0 and nd.value == 0
    assert L.pmp_debug_block_groups(handle.ptr, p, 8, 4624, 64, r, ctypes.byref(nd), None) == 0 and nd.value == 1


# ---- 2. outputs -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def loaded(exported):
    """(PartitionPredictor with the .pkl weights, two Handles with the same weights from .pmpw, their {qp: wsets[4]})."""
    pp = PartitionPredictor(0, engine="tc", chunk=4800)
    pp.load_pkls(MODELS, missing_bd="seeded")
    hs = [_lib.Handle(0) for _ in range(2)]
    ws = [{qp: [h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (c, t, qp))))[1] for c in COMPS for t in ("Q", "BD")]
           for qp in QPS} for h in hs]
    yield pp, hs, ws
    pp.close()
    for h in hs:
        h.close()


SHAPES = {"416x240_8bit": (416, 240, 6, 8, 4), "832x480_10bit": (832, 480, 5, 10, 2),
          "1080p_10bit": (1920, 1080, 4, 10, 3)}        # (width, height, frames, bit depth, uneven window)
KINDS = ["static", "letterbox", "flat", "tiled", "alias", "mixed"]


def _reference(pp, y, u, v):
    """{(comp index, qp): (values int8 [F*per], flags, qt, bt, dire)} of PartitionPredictor.predict_frames."""
    res = pp.predict_frames(y, u, v, qps=QPS, want_maps=True)
    return {(c, qp): (res[(comp, qp)][0].cpu().numpy().reshape(-1), res[(comp, qp)][4]) + res[(comp, qp)][1:4]
            for c, comp in enumerate(COMPS) for qp in QPS}


def _decoded(ref, c, qp, lamb, f, bh, bw):
    """The reference's maps decoded with `lamb` by the per-batch primitives: (values int8 [F*per], flags)."""
    _, _, qt, bt, dire = ref[(c, qp)]
    n = f * bh * bw
    _, qu8 = ops.qt_postprocess(qt, want_f32=False)
    hor, ver, dout, fl = ops.map2partition(qu8, bt, dire, 1 if c == 0 else 2, lamb=lamb, qt_raw=qt, near_tol=1e-2)
    return ops.assemble_frames(hor, ver, qu8.view(n, 64), dout, f, bh, bw).cpu().numpy().reshape(-1), fl


def _text(vals):
    return ops.format_text(torch.from_numpy(vals).cuda()).cpu().numpy().tobytes()


def _report_of(flag_list):
    tot = dict.fromkeys(REPORT_KEYS, 0)
    for fl in flag_list:
        for k, x in ops.flag_counts(fl).items():
            tot[k] += x
    return tot


def _check_stream(col, rep, want_vals, want_flags, text=True):
    for key, want in want_vals.items():
        got = np.concatenate(col.values[key])
        assert np.array_equal(got, want), key
        if text:
            assert b"".join(col.text[key]) == _text(want), key
    got = rep.as_dict()
    assert {k: got[k] for k in REPORT_KEYS} == _report_of(want_flags)
    assert got["fp16_saturation_events"] == 0


def _stats_reset(hs):
    for h in hs:
        h.block_stats(reset=True)


def _stats(hs):
    s = [h.block_stats() for h in hs]
    return sum(b for b, _ in s), sum(c for _, c in s)


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("kind", KINDS)
def test_outputs_are_byte_identical(loaded, kind, shape):
    pp, hs, ws = loaded
    wid, hgt, f, bd, window = SHAPES[shape]
    if kind == "alias" and bd == 8:
        pytest.skip("the 10-bit alias needs 10-bit samples")
    y, u, v = content(kind, wid, hgt, f, bd, seed=71 + KINDS.index(kind))
    bh, bw = hgt // 64, wid // 64
    bpf = bh * bw
    ref = _reference(pp, y, u, v)
    counts_w, counts_1 = distinct_counts(y, u, v, window), distinct_counts(y, u, v, 1)
    assert sum(dl for _, dl, _ in counts_w) < sum(n for n, _, _ in counts_w)      # the content has repeats
    h, w = hs[0], ws[0]

    # pmp_predict_host, QP 32, one-frame windows
    _stats_reset(hs)
    r = _lib.Report()
    got = h.predict_host(w[32], y, u, v, chunk=bpf, report=r)
    for c in range(2):
        assert np.array_equal(got[c].reshape(-1), ref[(c, 32)][0]), ("host", c)
    assert {k: r.as_dict()[k] for k in REPORT_KEYS} == _report_of([ref[(c, 32)][1] for c in range(2)])
    assert h.block_stats() == expected_stats(counts_1, 1)

    # pmp_predict_stream: all four QPs, values and text, uneven windows
    _stats_reset(hs)
    col = Collector(y, u, v)
    rep = h.predict_stream([w[qp] for qp in QPS], f, wid, hgt, y.itemsize, col.read, col.write, window_frames=window)
    _check_stream(col, rep, {(q, c): ref[(c, qp)][0] for q, qp in enumerate(QPS) for c in range(2)},
                  [ref[(c, qp)][1] for qp in QPS for c in range(2)])
    assert h.block_stats() == expected_stats(counts_w, len(QPS))

    # pmp_predict_stream_multi over two handles, one-frame windows in rotation
    _stats_reset(hs)
    col = Collector(y, u, v)
    rep = _lib.predict_stream_multi(hs, [[x[22], x[37]] for x in ws], f, wid, hgt, y.itemsize, col.read, col.write,
                                    window_frames=1)
    _check_stream(col, rep, {(q, c): ref[(c, qp)][0] for q, qp in enumerate((22, 37)) for c in range(2)},
                  [ref[(c, qp)][1] for qp in (22, 37) for c in range(2)])
    assert _stats(hs) == expected_stats(counts_1, 2)

    # pmp_predict_stream_ex: the four SWEEP threshold rows on one net pass, uneven windows
    _stats_reset(hs)
    col = Collector(y, u, v)
    rep = h.predict_stream([w[32]] * 4, f, wid, hgt, y.itemsize, col.read, col.write, window_frames=window, lamb=SWEEP)
    dec = {(r_, c): _decoded(ref, c, 32, lamb, f, bh, bw) for r_, lamb in enumerate(SWEEP) for c in range(2)}
    _check_stream(col, rep, {k: d[0] for k, d in dec.items()}, [d[1] for d in dec.values()])
    assert h.block_stats() == expected_stats(counts_w, 1)


# ---- 3. the work counted -------------------------------------------------------------------------------------------------
def _profiled(h, run):
    h.profile(2)                    # reset the counters and enable them
    run()
    got = h.profile_read()
    h.profile(0)
    return got


def test_work_scales_with_distinct_blocks(loaded):
    pp, hs, ws = loaded
    h, w = hs[0], ws[0]
    wid, hgt, f = 832, 480, 8
    runs = {}
    for kind in ("static", "letterbox", "mixed", "natural"):
        seqs = {kind: content(kind, wid, hgt, f, 10, seed=81)}
        seqs[kind + "_twin"] = perturbed(*seqs[kind])
        for name, (y, u, v) in seqs.items():
            counts = distinct_counts(y, u, v, 8)
            _stats_reset(hs)
            col = Collector(y, u, v)
            prof = _profiled(h, lambda: h.predict_stream([w[27]], f, wid, hgt, 2, col.read, col.write, window_frames=8))
            runs[name] = (h.block_stats(), prof, counts)
            assert runs[name][0] == expected_stats(counts, 1), name
    for name, ((blocks, computed), prof, _) in runs.items():
        if name.endswith("_twin") or name == "natural":
            assert computed == blocks, name             # the twins' blocks all differ
    for kind in ("static", "letterbox", "mixed"):
        (b, c), prof, _ = runs[kind]
        (bt, ct), prof_t, _ = runs[kind + "_twin"]
        assert c < b and bt == b == ct
        assert prof["conv_tc"]["flops"] == pytest.approx(prof_t["conv_tc"]["flops"] * c / ct, rel=1e-9), kind
    (b, c), _, _ = runs["static"]
    assert c <= b / 8                                   # 8 static frames in one window


def test_natural_content_runs_the_unchanged_sequence(loaded):
    """Without repeats nothing is gathered or expanded: the launch counts of the nets, the decode and the assembly equal
    those of ops.run_component over the same windows with the same chunk size."""
    pp, hs, ws = loaded
    h, w = hs[0], ws[0]
    y, u, v = synth.synth_yuv420(832, 480, 5, seed=82)
    bh, bw = 480 // 64, 832 // 64
    _stats_reset(hs)
    col = Collector(y, u, v)
    got = _profiled(h, lambda: h.predict_stream([w[32]], 5, 832, 480, 2, col.read, col.write, window_frames=2))
    blocks, computed = h.block_stats()
    assert computed == blocks == 2 * 5 * bh * bw
    lb, cb = ops.cut_blocks(_cuda(y), _cuda(u), _cuda(v))

    def reference():
        for f0 in range(0, 5, 2):
            nf = min(2, 5 - f0)
            sl = slice(f0 * bh * bw, (f0 + nf) * bh * bw)
            for c, blk in enumerate((lb, cb)):
                ops.run_component(w[32][2 * c], w[32][2 * c + 1], c == 0, blk[sl], nf, bh, bw, chunk=4800, handle=h)

    want = _profiled(h, reference)
    for cls in ("conv_tc", "decode", "assemble_frames"):
        assert got[cls]["launches"] == want[cls]["launches"] > 0, cls


# ---- 4. the saturation stop -----------------------------------------------------------------------------------------------
def test_saturation_stop_on_repeated_blocks(exported):
    h = _lib.Handle(0)
    try:
        wq = h.weights_create("Luma_Q", list(_saturating_luma_q().values()))
        _, wb = h.weights_load(str(exported / "Luma_BD_32.pmpw"))
        y, u, v = content("static", 256, 128, 6, 8, seed=1)
        col = Collector(y, u, v)
        rep = _lib.Report()
        with pytest.raises(_lib.PmpError) as e:
            h.predict_stream([[wq, wb, -1, -1]], 6, 256, 128, 1, col.read, col.write, window_frames=2, report=rep)
        assert "error -4" in str(e.value) and "PMP_TC_BF16" in str(e.value)
        assert [x[:2] for x in col.windows] == [(0, 2)]          # stopped after the first window
        assert rep.fp16_saturation_events > 0 and rep.blocks == 16
        blocks, computed = h.block_stats()
        assert blocks % 16 == 0 and 2 * computed == blocks       # the repeated frame of each window was not computed
    finally:
        h.close()


# ---- 5. the native tool -----------------------------------------------------------------------------------------------------
def _reuse_line(stdout):
    return [ln for ln in stdout.splitlines() if ln.startswith("Block reuse:")]


def test_native_tool_on_letterbox(loaded, exported, native_tool, tmp_path):
    pp = loaded[0]
    y, u, v = content("letterbox", 416, 240, 6, 10, seed=91)
    inp = tmp_path / "in"
    inp.mkdir()
    name = "seqL_416x240_10bit.yuv"
    _write_yuv(inp / name, y, u, v)
    (tmp_path / "seqs.txt").write_text("seqL,%s,416,240,6,1\n#end!!!!\n" % name)
    args = Inference_QBD.build_parser().parse_args([
        "--jobID", "j", "--inputDir", str(inp), "--outDir", str(tmp_path / "py"), "--batchSize", "200", "--seqNum", "1",
        "--seqInfo", str(tmp_path / "seqs.txt"), "--cfgDir", str(tmp_path / "nocfg"), "--modelDir", MODELS, "--ssRatio", "1",
        "--missingBD", "seeded", "--gpus", "1", "--binaryOut"])
    Inference_QBD.inference_VVC_seqs(args)
    py_dir = tmp_path / "py" / "j" / "PartitionMat"
    files = sorted(os.listdir(py_dir))
    assert len(files) == 16
    # the decode report of the same frames through the csrc/ path
    ref = _reference(pp, y, u, v)
    tot = _report_of([ref[k][1] for k in ref])
    want_report = ["Decode report: %d block-QPs, %d float32 near-tie argmins, %d with a map value within 0.01 of a decision "
                   "threshold (%d within 0.0001), 0 fp16 saturation events" % tuple(tot[k] for k in REPORT_KEYS)]
    for mode, extra, wf in (("default", (), 6), ("stream", ("--stream", "--chunk", "36"), 2)):
        out = tmp_path / mode
        r = subprocess.run([native_tool, "--input", str(inp / name), "--width", "416", "--height", "240", "--frames", "6",
                            "--bitDepth", "10", "--modelDir", str(exported), "--outDir", str(out), "--binaryOut", *extra],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        for n in files:
            assert open(py_dir / n, "rb").read() == open(out / n, "rb").read(), (mode, n)
        assert _report_line(r.stdout) == want_report, mode
        blocks, computed = expected_stats(distinct_counts(y, u, v, wf), len(QPS))
        assert computed < blocks
        assert _reuse_line(r.stdout) == ["Block reuse: the nets ran on %d of %d blocks (%.1f %%)" % (
            computed, blocks, 100.0 * computed / blocks)], (mode, r.stdout)


# ---- 6. distinct devices ------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more visible GPUs")
def test_reuse_on_distinct_devices(exported):
    hs = [_lib.Handle(d) for d in (0, 1)]
    try:
        ws = [[[h.weights_load(str(exported / ("%s_%s_32.pmpw" % (c, t))))[1] for c in COMPS for t in ("Q", "BD")]]
              for h in hs]
        y, u, v = content("mixed", 832, 480, 6, 10, seed=92)
        ref = Collector(y, u, v)
        want = hs[0].predict_stream(ws[0], 6, 832, 480, 2, ref.read, ref.write, window_frames=2)
        _stats_reset(hs)
        col = Collector(y, u, v)
        rep = _lib.predict_stream_multi(hs, ws, 6, 832, 480, 2, col.read, col.write, window_frames=2)
        assert {k: np.concatenate(a).tobytes() for k, a in col.values.items()} == \
            {k: np.concatenate(a).tobytes() for k, a in ref.values.items()}
        assert {k: b"".join(a) for k, a in col.text.items()} == {k: b"".join(a) for k, a in ref.text.items()}
        assert rep.as_dict() == want.as_dict()
        assert _stats(hs) == expected_stats(distinct_counts(y, u, v, 2), 1)
        assert all(h.block_stats()[0] > 0 for h in hs)
    finally:
        for h in hs:
            h.close()
