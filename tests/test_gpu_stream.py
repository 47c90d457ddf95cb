"""Streaming a sequence to PartitionMat data on the GPU: the batched asynchronous text kernel (pmp_format_texts) against
ops.format_text, pmp_predict_stream against pmp_predict_host window by window, its callbacks, errors, saturation and
bounded staging, and the native tool's --stream path against its default path."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from pmp_vvc_tip2023_b200 import _lib, build, export_weights, ops, synth, weights
from pmp_vvc_tip2023_b200.netspec import QPS
from tests import cases

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
MODELS = os.path.join(ROOT, "trained_models")
COMPS = ("Luma", "Chroma")
TILE = 4096         # values per CTA of pmp_format_texts_kernel


@pytest.fixture(scope="module")
def exported(tmp_path_factory):
    out = tmp_path_factory.mktemp("pmpw")
    export_weights.export(MODELS, str(out), missing_bd="seeded")
    return out


@pytest.fixture(scope="module")
def native_tool(tmp_path_factory):
    return build.build_native_tool(str(tmp_path_factory.mktemp("native") / "pmp_predict"))


@pytest.fixture(scope="module")
def loaded(exported):
    """A Handle with every QP's weight sets from the .pmpw files: (handle, {qp: wsets[4]})."""
    h = _lib.Handle(0)
    ws = {qp: [h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (c, t, qp))))[1] for c in COMPS for t in ("Q", "BD")]
          for qp in QPS}
    yield h, ws
    h.close()


# ---- pmp_format_texts -------------------------------------------------------------------------------------------------
def _vector(n, kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "all_neg":
        a = np.full(n, -1, np.int8)
    elif kind == "no_neg":
        a = rng.integers(0, 4, n).astype(np.int8)
    else:
        a = rng.integers(-1, 4, n).astype(np.int8)
    return torch.from_numpy(a).cuda()


def _format_texts(h, vecs, stream=0, text_offset=0):
    """pmp_format_texts over device int8 vectors; returns (texts, n_bytes) as device tensors, without synchronising."""
    m = len(vecs)
    bufs = [torch.full((3 * v.numel() + text_offset + 16,), 0xAA, dtype=torch.uint8, device="cuda") for v in vecs]
    nb = torch.full((m,), -7, dtype=torch.int64, device="cuda")
    vals = (ctypes.c_void_p * m)(*[v.data_ptr() if v.numel() else None for v in vecs])
    n = (ctypes.c_int64 * m)(*[v.numel() for v in vecs])
    txt = (ctypes.c_void_p * m)(*[b.data_ptr() + text_offset for b in bufs])
    _lib.check(_lib.lib().pmp_format_texts(h.ptr, m, vals, n, txt, ctypes.c_void_p(nb.data_ptr()),
                                           ctypes.c_void_p(stream)))
    return [b[text_offset:] for b in bufs], nb


def _check_texts(vecs, bufs, nb):
    nb = nb.cpu().tolist()
    for v, b, k in zip(vecs, bufs, nb):
        want = ops.format_text(v).cpu()
        assert k == want.numel()
        assert torch.equal(b[:k].cpu(), want)
        assert (b[k:k + 16].cpu() == 0xAA).all()          # nothing beyond the counted bytes


@pytest.mark.parametrize("kind", ["all_neg", "no_neg", "random"])
@pytest.mark.parametrize("n", [0, 1, TILE - 1, TILE, TILE + 1, 10 ** 7 + 13])
def test_format_texts_one_vector(n, kind):
    h = _lib.Handle(0)
    v = _vector(n, kind, seed=n % 1000)
    bufs, nb = _format_texts(h, [v])
    torch.cuda.synchronize()
    _check_texts([v], bufs, nb)
    h.close()


def test_format_texts_eight_vectors_one_launch():
    """Different lengths (empty ones among them), a value vector at an odd address and text at an odd address."""
    h = _lib.Handle(0)
    lens = [3 * TILE + 5, 0, 1, 70001, TILE, 0, 123457, 2 * TILE - 1]
    vecs = [_vector(n, ("random", "all_neg", "no_neg")[i % 3], seed=40 + i) for i, n in enumerate(lens)]
    vecs[3] = _vector(70004, "random", seed=99)[3:]            # 3 bytes past an aligned allocation
    launches = h.launch_count()
    bufs, nb = _format_texts(h, vecs, text_offset=5)
    assert h.launch_count() == launches + 1
    torch.cuda.synchronize()
    _check_texts(vecs, bufs, nb)
    bufs, nb = _format_texts(h, [torch.empty(0, dtype=torch.int8, device="cuda")] * 3)     # all empty
    torch.cuda.synchronize()
    assert nb.cpu().tolist() == [0, 0, 0]
    h.close()


def test_format_texts_does_not_synchronise():
    """Queued behind a long kernel on a side stream, the call returns before its work ran; the results are read only
    after an event recorded later on that stream."""
    h = _lib.Handle(0)
    vecs = [_vector(2 * 10 ** 6 + 1, "random", seed=5), _vector(777, "all_neg", seed=6)]
    s = torch.cuda.Stream()
    _format_texts(h, vecs)                                 # the first call of a handle allocates its status words
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)                     # ~0.1 s of GPU time before the text launch
        bufs, nb = _format_texts(h, vecs, stream=s.cuda_stream)
        done = torch.cuda.Event()
        done.record(s)
    assert not done.query()
    done.synchronize()
    _check_texts(vecs, bufs, nb)
    h.close()


def test_format_texts_bad_arguments():
    h = _lib.Handle(0)
    L = _lib.lib()
    v = _vector(10, "random", seed=1)
    nb = torch.zeros(9, dtype=torch.int64, device="cuda")
    t = torch.empty(30, dtype=torch.uint8, device="cuda")
    for m, n in ((0, 10), (9, 10), (1, -1), (1, (1 << 30) + 1)):
        k = max(m, 1)
        vals = (ctypes.c_void_p * k)(*([v.data_ptr()] * k))
        txt = (ctypes.c_void_p * k)(*([t.data_ptr()] * k))
        rc = L.pmp_format_texts(h.ptr, m, vals, (ctypes.c_int64 * k)(*([n] * k)), txt, ctypes.c_void_p(nb.data_ptr()),
                                None)
        assert rc == -1, (m, n)
    h.close()


# ---- pmp_predict_stream against pmp_predict_host -----------------------------------------------------------------------
class Collector:
    """read/write callbacks over host planes; keeps copies of every window's results."""

    def __init__(self, y, u, v, fail_read_at=None, fail_write_at=None):
        self.y, self.u, self.v = y, u, v
        self.reads, self.windows = [], []
        self.values, self.text = {}, {}
        self.fail_read_at, self.fail_write_at = fail_read_at, fail_write_at

    def read(self, f0, nf, y, u, v):
        self.reads.append((f0, nf, u is None))
        if len(self.reads) - 1 == self.fail_read_at:
            return 3
        y[...] = self.y[f0:f0 + nf]
        if u is not None:
            u[...] = self.u[f0:f0 + nf]
            v[...] = self.v[f0:f0 + nf]
        return 0

    def write(self, w):
        if len(self.windows) == self.fail_write_at:
            self.windows.append((w.first_frame, w.frames, w.report))
            return 5
        self.windows.append((w.first_frame, w.frames, w.report))
        for k, a in w.values.items():
            self.values.setdefault(k, []).append(a.copy())
        for k, a in w.text.items():
            self.text.setdefault(k, []).append(a.tobytes())
        return 0


def _stream_case(name):
    """(y, u, v, qps, {qp index: skipped component or None}, window_frames)."""
    if name == "pipe_192x128_10bit":
        y, u, v = cases.pipeline_frames()
        return y, u, v, (32,), {}, 0
    if name == "416x240_8bit_all_qps_window1":
        return synth.synth_yuv420(416, 240, 3, seed=31, bitdepth=8) + (QPS, {}, 1)
    if name == "832x480_10bit_window2_of_5":
        return synth.synth_yuv420(832, 480, 5, seed=32) + ((27, 37), {}, 2)
    if name == "1080p_10bit_3f_default":
        return synth.synth_yuv420(1920, 1080, 3, seed=33) + ((22, 32), {}, 0)
    if name == "416x240_8bit_luma_only":
        return synth.synth_yuv420(416, 240, 4, seed=34, bitdepth=8) + ((22, 37), {0: "Chroma", 1: "Chroma"}, 3)
    if name == "416x240_10bit_chroma_only":
        return synth.synth_yuv420(416, 240, 4, seed=35) + ((27,), {0: "Luma"}, 3)
    if name == "416x240_8bit_mixed":
        return synth.synth_yuv420(416, 240, 3, seed=36, bitdepth=8) + ((22, 32, 37), {0: "Chroma", 2: "Luma"}, 2)
    raise KeyError(name)


def _rows(ws, qps, skip):
    rows = []
    for i, qp in enumerate(qps):
        r = list(ws[qp])
        if skip.get(i) == "Luma":
            r[0:2] = [-1, -1]
        elif skip.get(i) == "Chroma":
            r[2:4] = [-1, -1]
        rows.append(r)
    return rows


@pytest.mark.parametrize("name", ["pipe_192x128_10bit", "416x240_8bit_all_qps_window1", "832x480_10bit_window2_of_5",
                                  "1080p_10bit_3f_default", "416x240_8bit_luma_only", "416x240_10bit_chroma_only",
                                  "416x240_8bit_mixed"])
def test_stream_equals_predict_host(loaded, name):
    h, ws = loaded
    y, u, v, qps, skip, window = _stream_case(name)
    f, hgt, wid = y.shape
    rows = _rows(ws, qps, skip)
    col = Collector(y, u, v)
    rep = h.predict_stream(rows, f, wid, hgt, y.itemsize, col.read, col.write, window_frames=window)
    # windows tile [0, frames) in order, each read once before it is written
    wf = window if window > 0 else max(1, 4800 // ((hgt // 64) * (wid // 64)))
    starts = list(range(0, f, wf))
    assert [(a, b) for a, b, _ in col.windows] == [(s, min(wf, f - s)) for s in starts]
    chroma = any(r[2] != -1 for r in rows)
    assert col.reads == [(s, min(wf, f - s), not chroma) for s in starts]
    want_rep = dict.fromkeys(rep.as_dict(), 0)
    for i, (qp, row) in enumerate(zip(qps, rows)):
        r = _lib.Report()
        got = h.predict_host(row, y, u if row[2] != -1 else None, v if row[2] != -1 else None, report=r)
        for k, n in r.as_dict().items():
            want_rep[k] += n
        for c in range(2):
            if got[c] is None:
                assert (i, c) not in col.values and (i, c) not in col.text
                continue
            vals = np.concatenate(col.values[(i, c)])
            assert np.array_equal(vals, got[c].reshape(-1)), (name, qp, c)
            text = b"".join(col.text[(i, c)])
            assert text == ops.format_text(torch.from_numpy(got[c]).cuda()).cpu().numpy().tobytes(), (name, qp, c)
            if name == "pipe_192x128_10bit":
                assert text == open(os.path.join(GOLDEN, "pipeline_%s_QP32_PartitionMat.txt" % COMPS[c]), "rb").read()
    assert rep.as_dict() == want_rep
    summed = dict.fromkeys(want_rep, 0)
    for _, _, r in col.windows:
        for k, n in r.items():
            summed[k] += n
    assert summed == want_rep and want_rep["fp16_saturation_events"] == 0
    print(name, want_rep)


@pytest.mark.parametrize("outputs", [_lib.OUT_VALUES, _lib.OUT_TEXT])
def test_stream_one_output_kind(loaded, outputs):
    h, ws = loaded
    y, u, v = synth.synth_yuv420(416, 240, 2, seed=37, bitdepth=8)
    col = Collector(y, u, v)
    h.predict_stream([ws[32]], 2, 416, 240, 1, col.read, col.write, outputs=outputs)
    got = h.predict_host(ws[32], y, u, v)
    assert bool(col.values) == (outputs == _lib.OUT_VALUES) and bool(col.text) == (outputs == _lib.OUT_TEXT)
    for c in range(2):
        if outputs == _lib.OUT_VALUES:
            assert np.array_equal(np.concatenate(col.values[(0, c)]), got[c].reshape(-1))
        else:
            assert b"".join(col.text[(0, c)]) == ops.format_text(torch.from_numpy(got[c]).cuda()).cpu().numpy().tobytes()


# ---- callbacks and errors -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["read", "write"])
def test_stream_callback_failure_aborts(loaded, which):
    h, ws = loaded
    y, u, v = synth.synth_yuv420(416, 240, 6, seed=38, bitdepth=8)
    col = Collector(y, u, v, **{"fail_%s_at" % which: 2})
    with pytest.raises(_lib.PmpError, match=r"error -6: the %s callback returned %d" % (which, 3 if which == "read" else 5)):
        h.predict_stream([ws[22], ws[37]], 6, 416, 240, 1, col.read, col.write, window_frames=1)
    if which == "read":
        assert len(col.reads) == 3 and all(w[0] < 2 for w in col.windows)
    else:
        assert [w[0] for w in col.windows] == [0, 1, 2]
    # the handle is still usable and right
    got = h.predict_host(ws[22], y, u, v)
    again = Collector(y, u, v)
    h.predict_stream([ws[22]], 6, 416, 240, 1, again.read, again.write, window_frames=4)
    for c in range(2):
        assert np.array_equal(np.concatenate(again.values[(0, c)]), got[c].reshape(-1))


def test_stream_python_exception_is_reraised(loaded):
    h, ws = loaded
    y, u, v = synth.synth_yuv420(256, 128, 3, seed=39, bitdepth=8)
    col = Collector(y, u, v)

    def bad_write(w):
        if w.first_frame == 1:
            raise ValueError("disk full")
        return col.write(w)

    with pytest.raises(ValueError, match="disk full") as e:
        h.predict_stream([ws[32]], 3, 256, 128, 1, col.read, bad_write, window_frames=1)
    assert isinstance(e.value.__context__, _lib.PmpError) and "-6" in str(e.value.__context__)
    assert [w[0] for w in col.windows] == [0]


def test_stream_bad_arguments_call_nothing(loaded):
    h, ws = loaded
    L = _lib.lib()
    calls = []
    rd = _lib.READ_CB(lambda *a: calls.append("read") or 0)
    wr = _lib.WRITE_CB(lambda *a: calls.append("write") or 0)
    good = list(ws[32])

    def call(rows, n_qps=None, frames=2, width=256, height=128, sb=1, outputs=3, read=rd, write=wr):
        flat = (ctypes.c_int * 16)(*(sum(rows, []) + [0] * (16 - 4 * len(rows))))
        return L.pmp_predict_stream(h.ptr, len(rows) if n_qps is None else n_qps, flat, frames, width, height, sb, 0,
                                    outputs, read, write, None, None)

    assert call([good]) == 0 and calls == ["read", "write"]
    calls.clear()
    bad = [dict(rows=[good], n_qps=0), dict(rows=[good] * 4, n_qps=5), dict(rows=[[good[1], good[0]] + good[2:]]),
           dict(rows=[good, [-1, -1, -1, -1]]), dict(rows=[good], outputs=0), dict(rows=[good], outputs=4),
           dict(rows=[good], read=_lib.READ_CB()), dict(rows=[good], write=_lib.WRITE_CB()), dict(rows=[good], width=255),
           dict(rows=[good], sb=3), dict(rows=[good], frames=-1)]
    for kw in bad:
        assert call(**kw) == -1, kw
    assert calls == []
    assert call([good], width=62) == 0 and call([good], frames=0) == 0 and calls == []


# ---- saturation -----------------------------------------------------------------------------------------------------
def _saturating_luma_q():
    sdq = synth.seeded_state_dict("Luma_Q", 3)     # the weights of test_fp16_saturation_is_reported
    return {k: v * 2000.0 if k.startswith("resblock_q1.left.0") else v for k, v in sdq.items()}


def test_stream_stops_after_saturating_window(exported):
    h = _lib.Handle(0)
    wq = h.weights_create("Luma_Q", list(_saturating_luma_q().values()))
    _, wb = h.weights_load(str(exported / "Luma_BD_32.pmpw"))
    y, u, v = synth.synth_yuv420(256, 128, 5, seed=1, bitdepth=8)
    col = Collector(y, u, v)
    before = h.saturation_count()
    rep = _lib.Report()
    with pytest.raises(_lib.PmpError) as e:
        h.predict_stream([[wq, wb, -1, -1]], 5, 256, 128, 1, col.read, col.write, window_frames=1, report=rep)
    assert "error -4" in str(e.value) and "PMP_TC_BF16" in str(e.value)
    events = [w[2]["fp16_saturation_events"] for w in col.windows]
    assert events[-1] > 0 and all(n == 0 for n in events[:-1])     # written up to the first saturating window only
    assert [w[0] for w in col.windows] == list(range(len(events)))
    assert rep.fp16_saturation_events == sum(events) and rep.blocks == 8 * len(events)
    assert h.saturation_count() >= before + rep.fp16_saturation_events
    h.close()


# ---- bounded staging --------------------------------------------------------------------------------------------------
def test_stream_memory_does_not_grow_with_frames(exported):
    h = _lib.Handle(0)
    rows = [[h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (c, t, qp))))[1] for c in COMPS for t in ("Q", "BD")]
            for qp in QPS]
    y, u, v = synth.synth_yuv420(416, 240, 40, seed=41, bitdepth=8)

    def run(f):
        col = Collector(y, u, v)
        h.predict_stream(rows, f, 416, 240, 1, col.read, lambda w: 0, window_frames=2)

    run(4)
    torch.cuda.synchronize()
    free4 = torch.cuda.mem_get_info()[0]
    run(40)
    torch.cuda.synchronize()
    free40 = torch.cuda.mem_get_info()[0]
    h.close()
    assert abs(free4 - free40) <= 8 << 20, (free4, free40)


# ---- the native tool's --stream path --------------------------------------------------------------------------------
def _write_yuv(path, y, u, v):
    with open(path, "wb") as fp:
        for f in range(y.shape[0]):
            fp.write(y[f].tobytes()); fp.write(u[f].tobytes()); fp.write(v[f].tobytes())


def _tool(tool, seq, w, hgt, frames, models, out, *extra):
    cmd = [tool, "--input", str(seq), "--width", str(w), "--height", str(hgt), "--frames", str(frames), "--modelDir",
           str(models), "--outDir", str(out)] + list(extra)
    return subprocess.run(cmd, capture_output=True, text=True)


def _report_line(stdout):
    return [ln for ln in stdout.splitlines() if ln.startswith("Decode report:")]


def test_native_tool_stream_matches_default_path(exported, native_tool, tmp_path):
    y, u, v = cases.pipeline_frames()
    seq = tmp_path / "pipe_192x128_10bit.yuv"
    _write_yuv(seq, y, u, v)
    args = ("--bitDepth", "10", "--qps", "32", "--binaryOut")
    ref = _tool(native_tool, seq, 192, 128, cases.PIPE_F, exported, tmp_path / "a", *args)
    got = _tool(native_tool, seq, 192, 128, cases.PIPE_F, exported, tmp_path / "b", *(args + ("--stream", "--timing")))
    print(got.stdout, got.stderr)
    assert ref.returncode == 0 and got.returncode == 0, got.stderr
    assert "pmp_predict_stream" in got.stdout and "(2 frames, 1 windows)" in got.stdout
    assert _report_line(ref.stdout) == _report_line(got.stdout)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(os.listdir(tmp_path / "b"))
    for n in os.listdir(tmp_path / "a"):
        assert open(tmp_path / "a" / n, "rb").read() == open(tmp_path / "b" / n, "rb").read(), n
    for comp in COMPS:
        want = open(os.path.join(GOLDEN, "pipeline_%s_QP32_PartitionMat.txt" % comp), "rb").read()
        assert open(tmp_path / "b" / ("pipe_192x128_10bit_%s_QP32_PartitionMat.txt" % comp), "rb").read() == want

    # 416x240, every 4th of 9 frames, all QPs, one-frame windows (--chunk 20, 18 blocks per frame)
    y, u, v = synth.synth_yuv420(416, 240, 9, seed=21, bitdepth=8)
    seq = tmp_path / "seqD_416x240_8bit.yuv"
    _write_yuv(seq, y, u, v)
    args = ("--ssRatio", "4", "--binaryOut")
    ref = _tool(native_tool, seq, 416, 240, 9, exported, tmp_path / "c", *args)
    got = _tool(native_tool, seq, 416, 240, 9, exported, tmp_path / "d", *(args + ("--stream", "--chunk", "20")))
    assert ref.returncode == 0 and got.returncode == 0, got.stderr
    assert _report_line(ref.stdout) == _report_line(got.stdout)
    files = sorted(os.listdir(tmp_path / "c"))
    assert len(files) == 16 and files == sorted(os.listdir(tmp_path / "d"))
    for n in files:
        assert open(tmp_path / "c" / n, "rb").read() == open(tmp_path / "d" / n, "rb").read(), n
    # without --binaryOut a stale .bin beside the new .txt is removed
    got = _tool(native_tool, seq, 416, 240, 9, exported, tmp_path / "d", "--ssRatio", "4", "--qps", "27", "--stream")
    assert got.returncode == 0, got.stderr
    left = sorted(os.listdir(tmp_path / "d"))
    assert "seqD_416x240_8bit_Luma_QP27_PartitionMat.bin" not in left and "seqD_416x240_8bit_Luma_QP22_PartitionMat.bin" in left
    assert len(left) == 14


def test_native_tool_stream_saturation_writes_nothing(exported, native_tool, tmp_path):
    models = tmp_path / "models"
    models.mkdir()
    weights.write_pmpw(str(models / "Luma_Q_32.pmpw"), "Luma_Q", _saturating_luma_q())
    for n in ("Luma_BD_32.pmpw", "Chroma_Q_32.pmpw", "Chroma_BD_32.pmpw"):
        shutil.copy(exported / n, models / n)
    y, u, v = synth.synth_yuv420(256, 128, 3, seed=1, bitdepth=8)
    seq = tmp_path / "sat_256x128.yuv"
    _write_yuv(seq, y, u, v)
    out = tmp_path / "out"
    out.mkdir()
    keep = out / "sat_256x128_Luma_QP32_PartitionMat.txt"
    keep.write_bytes(b"an earlier run\n")
    r = _tool(native_tool, seq, 256, 128, 3, models, out, "--qps", "32", "--stream", "--binaryOut", "--chunk", "8")
    print(r.stdout, r.stderr)
    assert r.returncode == 1 and "--tcDtype bf16" in r.stderr
    assert sorted(os.listdir(out)) == [keep.name] and keep.read_bytes() == b"an earlier run\n"
