"""PartitionMat data under several decode-threshold settings from one net pass (pmp_predict_stream_ex): every row against
an independent result (the nets' maps, the C oracle's post-process and decode with the row's lamb1..lamb5, assembled in
frame order), byte equality with pmp_predict_stream_multi for the default thresholds, mixed rows against one-row calls,
the shared net pass counted in launches, errors, the saturation stop and callback aborts with thresholds, the native
tool's --lamb, and handles on distinct devices."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import c_decode
from pmp_vvc_tip2023_b200 import _lib, ops, synth
from pmp_vvc_tip2023_b200.netspec import QPS
from tests import cases
from tests.test_gpu_stream import (COMPS, Collector, _saturating_luma_q, _tool, _write_yuv,  # noqa: F401
                                   exported, native_tool)

pytestmark = pytest.mark.gpu
DEFAULT = ops.DEFAULT_LAMB
SWEEP = [DEFAULT, cases.LAMB_SETS["a"], cases.LAMB_SETS["b"], cases.LAMB_SETS["c"]]


def _load_all(h, exported):
    """Every QP's weight sets from the .pmpw files on handle h: {qp: wsets[4]}."""
    return {qp: [h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (c, t, qp))))[1] for c in COMPS for t in ("Q", "BD")]
            for qp in QPS}


@pytest.fixture(scope="module")
def handles(exported):
    """Two handles on device 0, each with every QP's weights: ([handle], [{qp: wsets[4]}])."""
    hs = [_lib.Handle(0) for _ in range(2)]
    ws = [_load_all(h, exported) for h in hs]
    yield hs, ws
    for h in hs:
        h.close()


def _joined(col):
    return ({k: np.concatenate(v).tobytes() for k, v in col.values.items()},
            {k: b"".join(v) for k, v in col.text.items()})


def _cuda(a):
    return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda()


def _independent(h, wsets, y, u, v, lamb):
    """Per component: (values int8 [F * per] decoded by the C oracle from the nets' own maps with `lamb`, the same
    from the GPU decode kernel, and the block id of every value of blocks whose GPU decode flagged a float32 near-tie)."""
    f, hgt, wid = y.shape
    bh, bw = hgt // 64, wid // 64
    blocks = ops.cut_blocks(_cuda(y), _cuda(u), _cuda(v), handle=h)
    out = {}
    for c in range(2):
        cf = 1 if c == 0 else 2
        _, qt, bt, dire, _ = ops.run_component(wsets[2 * c], wsets[2 * c + 1], c == 0, blocks[c], f, bh, bw, chunk=4800,
                                               want_maps=True, handle=h)
        qi = c_decode.qt_postprocess(qt.cpu().numpy())[:, 0]
        hor, ver, dout = c_decode.map_to_partition_batch(qi, bt.cpu().numpy(), dire.cpu().numpy(), cf, lamb=lamb)
        n = f * bh * bw
        H = hor.reshape(f, bh, bw, 16, 16).transpose(0, 1, 3, 2, 4).reshape(f, -1)
        V = ver.reshape(f, bh, bw, 16, 16).transpose(0, 1, 3, 2, 4).reshape(f, -1)
        Q = qi.astype(np.int8).reshape(f, bh, bw, 8, 8).transpose(0, 1, 3, 2, 4).reshape(f, -1)
        D = dout.reshape(f, bh, bw, 3, 16, 16).transpose(0, 3, 1, 4, 2, 5).reshape(f, -1)
        want = np.concatenate([H, V, Q, D], axis=1).astype(np.int8).reshape(-1)
        _, qu8 = ops.qt_postprocess(qt, want_f32=False, handle=h)
        gh, gv, gd, fl = ops.map2partition(qu8, bt, dire, cf, lamb=lamb, qt_raw=qt, near_tol=1e-2, handle=h)
        gpu = ops.assemble_frames(gh, gv, qu8.view(n, 64), gd, f, bh, bw, handle=h).cpu().numpy().reshape(-1)
        tie = np.nonzero(fl.cpu().numpy() & 1)[0]
        out[c] = (want, gpu, tie)
    return out


def _lamb_case(name):
    """(y, u, v, window_frames)."""
    if name == "416x240_8bit_window1":
        return synth.synth_yuv420(416, 240, 3, seed=51, bitdepth=8) + (1,)
    if name == "832x480_10bit_window2_of_5":
        return synth.synth_yuv420(832, 480, 5, seed=52) + (2,)
    if name == "1080p_10bit_window2_of_3":
        return synth.synth_yuv420(1920, 1080, 3, seed=53) + (2,)
    if name == "1080p_8bit_one_frame":
        return synth.synth_yuv420(1920, 1080, 1, seed=54, bitdepth=8) + (0,)
    raise KeyError(name)


@pytest.mark.parametrize("n", [1, 2])
@pytest.mark.parametrize("name", ["416x240_8bit_window1", "832x480_10bit_window2_of_5", "1080p_10bit_window2_of_3",
                                  "1080p_8bit_one_frame"])
def test_rows_equal_independent_decode(handles, name, n):
    hs, ws = handles
    y, u, v, window = _lamb_case(name)
    f, hgt, wid = y.shape
    bh, bw = hgt // 64, wid // 64
    col = Collector(y, u, v)
    rep = _lib.predict_stream_multi(hs[:n], [[w[32]] * 4 for w in ws[:n]], f, wid, hgt, y.itemsize, col.read, col.write,
                                    window_frames=window, lamb=SWEEP)
    vals, text = _joined(col)
    assert sorted(vals) == sorted(text) == [(r, c) for r in range(4) for c in range(2)]
    ids = cases.value_block_ids(f, bh, bw)
    ties = 0
    for r, lamb in enumerate(SWEEP):
        ind = _independent(hs[0], ws[0][32], y, u, v, lamb)
        for c in range(2):
            want, gpu, tie = ind[c]
            got = np.frombuffer(vals[(r, c)], np.int8).copy()
            assert np.array_equal(got, gpu), (name, n, r, c)          # the per-batch primitives on the same maps
            diff = np.nonzero(got != want)[0]
            assert np.isin(ids[diff], tie).all(), (name, r, c, np.unique(ids[diff]))    # the oracle, but for near-ties
            ties += tie.size
            assert text[(r, c)] == ops.format_text(torch.from_numpy(got).cuda()).cpu().numpy().tobytes(), (name, r, c)
    assert rep.blocks == 4 * 2 * f * bh * bw and rep.near_tie_blocks == ties
    # the settings decode differently: the sweep is not four copies of one result
    assert len({vals[(r, 0)] for r in range(4)}) > 1


def test_default_thresholds_equal_stream_multi(handles):
    """lamb None, explicit default rows and pmp_predict_stream_multi are byte-identical, reports included."""
    hs, ws = handles
    y, u, v = synth.synth_yuv420(832, 480, 5, seed=55)
    rows = [[w[22], w[37]] for w in ws]
    runs = {}
    for key, lamb in (("multi", None), ("ex_defaults", [DEFAULT, DEFAULT])):
        col = Collector(y, u, v)
        rep = _lib.predict_stream_multi(hs, rows, 5, 832, 480, 2, col.read, col.write, window_frames=2, lamb=lamb)
        runs[key] = (_joined(col), rep.as_dict(), [w[:2] for w in col.windows])
    L = _lib.lib()
    col = Collector(y, u, v)
    rep = _lib.Report()
    flat = (ctypes.c_int * 16)(*[x for by in rows for r in by for x in r])
    hp = (ctypes.c_void_p * 2)(*[h.ptr for h in hs])
    _lib.check(L.pmp_predict_stream_ex(hp, 2, 2, flat, None, 5, 832, 480, 2, 2, 3, _lib.READ_CB(
        lambda _u, f0, nf, yy, uu, vv: _read_into(col, f0, nf, yy, uu, vv, 832, 480)), _lib.WRITE_CB(
        lambda _u, wp: col.write(_lib.StreamWindow(wp.contents, _view))), None, ctypes.byref(rep)))
    runs["ex_null"] = (_joined(col), rep.as_dict(), [w[:2] for w in col.windows])
    assert runs["ex_defaults"] == runs["multi"] and runs["ex_null"] == runs["multi"]
    # Handle.predict_stream with default rows equals pmp_predict_stream
    one = Collector(y, u, v)
    rep1 = hs[0].predict_stream(rows[0], 5, 832, 480, 2, one.read, one.write, window_frames=2)
    two = Collector(y, u, v)
    rep2 = hs[0].predict_stream(rows[0], 5, 832, 480, 2, two.read, two.write, window_frames=2, lamb=[DEFAULT] * 2)
    assert _joined(one) == _joined(two) and rep1.as_dict() == rep2.as_dict()


def _view(ptr, shape, dtype):
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    return np.frombuffer((ctypes.c_char * n).from_address(ptr), dtype).reshape(shape) if ptr else None


def _read_into(col, f0, nf, y, u, v, wid, hgt):
    dt = col.y.dtype
    return col.read(f0, nf, _view(y, (nf, hgt, wid), dt), _view(u, (nf, hgt // 2, wid // 2), dt),
                    _view(v, (nf, hgt // 2, wid // 2), dt))


def test_mixed_rows_equal_one_row_calls(handles):
    """Two QPs x two settings in one call: each row's bytes and the summed report equal four one-row calls."""
    hs, ws = handles
    h, w = hs[0], ws[0]
    y, u, v = synth.synth_yuv420(416, 240, 4, seed=56, bitdepth=8)
    a, b = cases.LAMB_SETS["a"], cases.LAMB_SETS["b"]
    rows = [(22, a), (22, b), (37, a), (37, b)]
    col = Collector(y, u, v)
    rep = h.predict_stream([w[qp] for qp, _ in rows], 4, 416, 240, 1, col.read, col.write, window_frames=3,
                           lamb=[l for _, l in rows])
    vals, text = _joined(col)
    want_rep = dict.fromkeys(rep.as_dict(), 0)
    for r, (qp, lamb) in enumerate(rows):
        one = Collector(y, u, v)
        r1 = h.predict_stream([w[qp]], 4, 416, 240, 1, one.read, one.write, window_frames=3, lamb=[lamb])
        ov, ot = _joined(one)
        for c in range(2):
            assert vals[(r, c)] == ov[(0, c)] and text[(r, c)] == ot[(0, c)], (r, c)
        for k, x in r1.as_dict().items():
            want_rep[k] += x
    assert rep.as_dict() == want_rep


def _launches(h, run):
    h.profile(2)                    # reset the counters and enable them
    run()
    got = {k: v["launches"] for k, v in h.profile_read().items()}
    h.profile(0)
    return got


def test_shared_weights_share_the_net_pass(handles):
    """Counted in launches, not time: four rows on one weight set launch the convolutions of one row and four times its
    decodes; four rows on four weight sets launch four times the convolutions."""
    hs, ws = handles
    h, w = hs[0], ws[0]
    y, u, v = synth.synth_yuv420(832, 480, 2, seed=57)

    def run(rows, lamb):
        col = Collector(y, u, v)
        return lambda: h.predict_stream(rows, 2, 832, 480, 2, col.read, col.write, window_frames=1, lamb=lamb)

    one = _launches(h, run([w[32]], [DEFAULT]))
    shared = _launches(h, run([w[32]] * 4, SWEEP))
    distinct = _launches(h, run([w[qp] for qp in QPS], SWEEP))
    assert one["conv_tc"] > 0 and one["decode"] > 0
    assert shared["conv_tc"] == one["conv_tc"] and shared["decode"] == 4 * one["decode"]
    assert shared["assemble_frames"] == 4 * one["assemble_frames"]
    assert distinct["conv_tc"] == 4 * one["conv_tc"] and distinct["decode"] == 4 * one["decode"]


# ---- errors -----------------------------------------------------------------------------------------------------------
def test_bad_thresholds_call_nothing(handles):
    hs, ws = handles
    L = _lib.lib()
    calls = []
    rd = _lib.READ_CB(lambda *a: calls.append("read") or 0)
    wr = _lib.WRITE_CB(lambda *a: calls.append("write") or 0)
    hp = (ctypes.c_void_p * 1)(hs[0].ptr)

    def call(lamb, n_rows=None):
        n_rows = len(lamb) if n_rows is None else n_rows
        flat = (ctypes.c_int * (4 * max(n_rows, 1)))(*(ws[0][32] * max(n_rows, 1)))
        lam = (ctypes.c_double * (5 * max(len(lamb), 1)))(*[x for t in lamb for x in t])
        rc = L.pmp_predict_stream_ex(hp, 1, n_rows, flat, lam, 2, 256, 128, 1, 0, 3, rd, wr, None, None)
        return rc, L.pmp_last_error().decode()

    assert call([DEFAULT])[0] == 0 and calls == ["read", "write"]
    calls.clear()
    bad = list(cases.LAMB_SETS["a"])
    bad[2] = float("nan")
    rc, msg = call([DEFAULT, tuple(bad)])
    assert rc == -1 and "lamb[1][2]" in msg and "row 1" in msg and "finite" in msg, msg
    for x in (float("inf"), float("-inf")):
        rc, msg = call([(0.7, 0.7, 1.5, 0.3, x)])
        assert rc == -1 and "lamb[0][4]" in msg, msg
    rc, msg = call([DEFAULT] * 5)
    assert rc == -1 and "n_rows must be 1 to 4" in msg
    rc, msg = call([DEFAULT], n_rows=0)
    assert rc == -1 and "n_rows must be 1 to 4" in msg
    y, u, v = synth.synth_yuv420(256, 128, 2, seed=58, bitdepth=8)
    col = Collector(y, u, v)
    with pytest.raises(ValueError, match="tuple per row"):
        hs[0].predict_stream([ws[0][32]] * 2, 2, 256, 128, 1, col.read, col.write, lamb=[DEFAULT])
    with pytest.raises(_lib.PmpError, match="lamb\\[0\\]\\[0\\]"):
        hs[0].predict_stream([ws[0][32]], 2, 256, 128, 1, col.read, col.write, lamb=[(float("nan"),) + DEFAULT[1:]])
    assert calls == [] and col.reads == [] and col.windows == []


@pytest.mark.parametrize("which", ["read", "write"])
def test_callback_abort_with_thresholds(handles, which):
    hs, ws = handles
    y, u, v = synth.synth_yuv420(416, 240, 6, seed=59, bitdepth=8)
    col = Collector(y, u, v, **{"fail_%s_at" % which: 3 if which == "read" else 2})
    with pytest.raises(_lib.PmpError, match=r"error -6: the %s callback returned %d" % (which, 3 if which == "read" else 5)):
        _lib.predict_stream_multi(hs, [[w[22]] * 2 for w in ws], 6, 416, 240, 1, col.read, col.write, window_frames=1,
                                  lamb=SWEEP[:2])
    if which == "read":
        assert [r[0] for r in col.reads] == [0, 1, 2, 3] and all(w[0] < 3 for w in col.windows)
    else:
        assert [w[0] for w in col.windows] == [0, 1, 2]
    again = Collector(y, u, v)          # every handle is still usable
    _lib.predict_stream_multi(hs, [[w[22]] for w in ws], 6, 416, 240, 1, again.read, again.write, window_frames=4,
                              lamb=[DEFAULT])
    got = hs[0].predict_host(ws[0][22], y, u, v)
    for c in range(2):
        assert np.array_equal(np.concatenate(again.values[(0, c)]), got[c].reshape(-1))


def test_stops_after_saturating_window_with_thresholds(exported):
    sat = list(_saturating_luma_q().values())
    hs = [_lib.Handle(0) for _ in range(2)]
    try:
        rows = [[[h.weights_create("Luma_Q", sat), h.weights_load(str(exported / "Luma_BD_32.pmpw"))[1], -1, -1]] * 2
                for h in hs]
        y, u, v = synth.synth_yuv420(256, 128, 5, seed=1, bitdepth=8)
        single = Collector(y, u, v)
        with pytest.raises(_lib.PmpError, match="error -4"):
            _lib.predict_stream_multi(hs, [r[:1] for r in rows], 5, 256, 128, 1, single.read, single.write,
                                      window_frames=1)
        col = Collector(y, u, v)
        rep = _lib.Report()
        with pytest.raises(_lib.PmpError) as e:
            _lib.predict_stream_multi(hs, rows, 5, 256, 128, 1, col.read, col.write, window_frames=1, report=rep,
                                      lamb=[DEFAULT, cases.LAMB_SETS["c"]])
        assert "error -4" in str(e.value) and "PMP_TC_BF16" in str(e.value)
        events = [w[2]["fp16_saturation_events"] for w in col.windows]
        assert events[-1] > 0 and all(n == 0 for n in events[:-1])
        assert [w[:2] for w in col.windows] == [w[:2] for w in single.windows]
        assert rep.fp16_saturation_events == sum(events) and rep.blocks == 2 * 8 * len(events)
    finally:
        for h in hs:
            h.close()


# ---- the native tool's --lamb -----------------------------------------------------------------------------------------
def test_native_tool_lamb(handles, exported, native_tool, tmp_path):
    hs, ws = handles
    y, u, v = synth.synth_yuv420(416, 240, 3, seed=60)
    seq = tmp_path / "seqL_416x240_10bit.yuv"
    _write_yuv(seq, y, u, v)
    a, b = cases.LAMB_SETS["a"], cases.LAMB_SETS["b"]
    fmt = lambda t: ",".join(repr(x) for x in t)       # noqa: E731
    r = _tool(native_tool, seq, 416, 240, 3, exported, tmp_path / "two", "--bitDepth", "10", "--qps", "32", "--stream",
              "--lamb", fmt(a), "--lamb", fmt(b), "--binaryOut", "--timing")
    assert r.returncode == 0, r.stderr
    assert "pmp_predict_stream_ex" in r.stdout and "2 rows" in r.stdout
    assert "Thresholds of %s: lamb1..lamb5 = 0.6,0.8,1.2,0.4,0.6" % (tmp_path / "two" / "lamb0") in r.stdout
    assert "Thresholds of %s: lamb1..lamb5 = 0.9,0.5,2,0.2,0.8" % (tmp_path / "two" / "lamb1") in r.stdout
    assert sorted(os.listdir(tmp_path / "two")) == ["lamb0", "lamb1"]
    col = Collector(y, u, v)
    hs[0].predict_stream([ws[0][32]] * 2, 3, 416, 240, 2, col.read, col.write, lamb=[a, b])
    vals, text = _joined(col)
    for i in range(2):
        d = tmp_path / "two" / ("lamb%d" % i)
        assert len(os.listdir(d)) == 4
        for c, comp in enumerate(COMPS):
            stem = "seqL_416x240_10bit_%s_QP32_PartitionMat" % comp
            assert open(d / (stem + ".txt"), "rb").read() == text[(i, c)], (i, comp)
            assert open(d / (stem + ".bin"), "rb").read()[32:] == vals[(i, c)], (i, comp)
    assert text[(0, 0)] != text[(1, 0)]
    # one --lamb holding the defaults: the usual names in --outDir, byte-identical to a run without --lamb
    runs = {"plain": (), "defaults": ("--lamb", "0.7,0.7,1.5,0.3,0.7")}
    for k, extra in runs.items():
        r = _tool(native_tool, seq, 416, 240, 3, exported, tmp_path / k, "--bitDepth", "10", "--qps", "22,37",
                  "--stream", "--binaryOut", *extra)
        assert r.returncode == 0, r.stderr
    files = sorted(os.listdir(tmp_path / "plain"))
    assert len(files) == 8 and sorted(os.listdir(tmp_path / "defaults")) == files
    for n in files:
        assert open(tmp_path / "plain" / n, "rb").read() == open(tmp_path / "defaults" / n, "rb").read(), n


def test_native_tool_lamb_failure_replaces_nothing(exported, native_tool, tmp_path):
    """A run that fails (here: the sequence is shorter than --frames) leaves every directory as it was."""
    y, u, v = synth.synth_yuv420(256, 128, 2, seed=61, bitdepth=8)
    seq = tmp_path / "short_256x128.yuv"
    _write_yuv(seq, y, u, v)
    out = tmp_path / "out"
    (out / "lamb1").mkdir(parents=True)
    keep = out / "lamb1" / "short_256x128_Luma_QP32_PartitionMat.txt"
    keep.write_bytes(b"an earlier run\n")
    r = _tool(native_tool, seq, 256, 128, 4, exported, out, "--qps", "32", "--stream", "--chunk", "8",
              "--lamb", "0.7,0.7,1.5,0.3,0.7", "--lamb", "0.6,0.8,1.2,0.4,0.6")
    assert r.returncode == 1 and "fewer than 4 frames" in r.stderr, r.stderr
    assert sorted(os.listdir(out / "lamb0")) == [] and sorted(os.listdir(out / "lamb1")) == [keep.name]
    assert keep.read_bytes() == b"an earlier run\n"


# ---- distinct devices -------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more visible GPUs")
def test_lamb_rows_on_distinct_devices(exported):
    hs = [_lib.Handle(d) for d in (0, 1)]
    try:
        ws = [_load_all(h, exported) for h in hs]
        y, u, v = synth.synth_yuv420(832, 480, 5, seed=62)
        ref = Collector(y, u, v)
        want = hs[0].predict_stream([ws[0][27]] * 4, 5, 832, 480, 2, ref.read, ref.write, window_frames=2, lamb=SWEEP)
        col = Collector(y, u, v)
        rep = _lib.predict_stream_multi(hs, [[w[27]] * 4 for w in ws], 5, 832, 480, 2, col.read, col.write,
                                        window_frames=2, lamb=SWEEP)
        assert _joined(col) == _joined(ref) and rep.as_dict() == want.as_dict()
    finally:
        for h in hs:
            h.close()
