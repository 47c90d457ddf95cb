"""One sequence over several handles in one call (pmp_predict_stream_multi): byte equality with pmp_predict_stream on one
handle for 1, 2 and 3 handles on one device, callback order and thread, argument and consistency errors, callback
failures, the saturation stop, bounded staging, the native tool's --devices, and handles on distinct devices."""
import ctypes
import os
import threading

import numpy as np
import pytest
import torch

from pmp_vvc_tip2023_b200 import _lib, synth
from pmp_vvc_tip2023_b200.netspec import QPS
from tests import cases
from tests.test_gpu_stream import (COMPS, Collector, _report_line, _rows, _saturating_luma_q, _tool,  # noqa: F401
                                   _write_yuv, exported, native_tool)

pytestmark = pytest.mark.gpu
MAX_HANDLES = 3


def _load_all(h, exported):
    """Every QP's weight sets from the .pmpw files on handle h: {qp: wsets[4]}."""
    return {qp: [h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (c, t, qp))))[1] for c in COMPS for t in ("Q", "BD")]
            for qp in QPS}


@pytest.fixture(scope="module")
def handles(exported):
    """Three handles on device 0, each with every QP's weights: ([handle], [{qp: wsets[4]}])."""
    hs = [_lib.Handle(0) for _ in range(MAX_HANDLES)]
    ws = [_load_all(h, exported) for h in hs]
    yield hs, ws
    for h in hs:
        h.close()


class OrderCollector(Collector):
    """A Collector that also records the thread and the current device of every callback."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.threads, self.devices = set(), set()

    def read(self, f0, nf, y, u, v):
        self.threads.add(threading.get_ident())
        self.devices.add(torch.cuda.current_device())
        return super().read(f0, nf, y, u, v)

    def write(self, w):
        self.threads.add(threading.get_ident())
        self.devices.add(torch.cuda.current_device())
        return super().write(w)


def _multi_case(name):
    """(y, u, v, qps, {qp index: skipped component}, window_frames)."""
    if name == "416x240_8bit_all_qps_window1":
        return synth.synth_yuv420(416, 240, 3, seed=31, bitdepth=8) + (QPS, {}, 1)
    if name == "832x480_10bit_5f_window2":
        return synth.synth_yuv420(832, 480, 5, seed=32) + ((27, 37), {}, 2)
    if name == "1080p_10bit_window2_of_5":
        return synth.synth_yuv420(1920, 1080, 5, seed=33) + ((22, 32), {}, 2)
    if name == "416x240_8bit_single_component_row":
        return synth.synth_yuv420(416, 240, 4, seed=34, bitdepth=8) + ((22, 37), {1: "Chroma"}, 1)
    if name == "416x240_10bit_one_frame":
        return synth.synth_yuv420(416, 240, 1, seed=35) + ((32,), {}, 0)
    if name == "832x480_10bit_default_window":
        return synth.synth_yuv420(832, 480, 7, seed=36) + ((22, 27), {}, 0)
    raise KeyError(name)


def _joined(col):
    return ({k: np.concatenate(v).tobytes() for k, v in col.values.items()},
            {k: b"".join(v) for k, v in col.text.items()})


def _window_frames(window, frames, hgt, wid, n):
    bpf = (hgt // 64) * (wid // 64)
    return min(frames, window if window > 0 else max(1, min(4800 // bpf, -(-frames // n))))


_single = {}


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("name", ["416x240_8bit_all_qps_window1", "832x480_10bit_5f_window2", "1080p_10bit_window2_of_5",
                                  "416x240_8bit_single_component_row", "416x240_10bit_one_frame",
                                  "832x480_10bit_default_window"])
def test_multi_equals_single_handle_stream(handles, name, n):
    hs, ws = handles
    y, u, v, qps, skip, window = _multi_case(name)
    f, hgt, wid = y.shape
    if name not in _single:         # pmp_predict_stream on handles[0], the same window argument
        col = Collector(y, u, v)
        rep = hs[0].predict_stream(_rows(ws[0], qps, skip), f, wid, hgt, y.itemsize, col.read, col.write,
                                   window_frames=window)
        _single[name] = (_joined(col), rep.as_dict())
    (want_vals, want_text), want_rep = _single[name]
    col = OrderCollector(y, u, v)
    rep = _lib.predict_stream_multi(hs[:n], [_rows(ws[i], qps, skip) for i in range(n)], f, wid, hgt, y.itemsize,
                                    col.read, col.write, window_frames=window)
    vals, text = _joined(col)
    assert vals.keys() == want_vals.keys() and text.keys() == want_text.keys()
    for k in want_vals:
        assert vals[k] == want_vals[k], (name, n, k)
        assert text[k] == want_text[k], (name, n, k)
    assert rep.as_dict() == want_rep and want_rep["fp16_saturation_events"] == 0
    wf = _window_frames(window, f, hgt, wid, n)
    starts = list(range(0, f, wf))
    assert [(a, b) for a, b, _ in col.windows] == [(s, min(wf, f - s)) for s in starts]
    assert [(a, b) for a, b, _ in col.reads] == [(s, min(wf, f - s)) for s in starts]
    assert col.threads == {threading.get_ident()} and col.devices == {0}


def test_multi_default_window_reaches_every_handle(handles):
    """Three 416x240 frames over three handles: the default window is one frame, not 3 (4800 / 18 blocks)."""
    hs, ws = handles
    y, u, v = synth.synth_yuv420(416, 240, 3, seed=40, bitdepth=8)
    col = Collector(y, u, v)
    launches = [h.launch_count() for h in hs]
    _lib.predict_stream_multi(hs, [[w[32]] for w in ws], 3, 416, 240, 1, col.read, col.write)
    assert [w[:2] for w in col.windows] == [(0, 1), (1, 1), (2, 1)]
    assert all(h.launch_count() > n for h, n in zip(hs, launches))        # every handle ran a window


# ---- callbacks ------------------------------------------------------------------------------------------------------
def test_multi_callback_order_and_thread(handles):
    hs, ws = handles
    y, u, v = synth.synth_yuv420(256, 128, 11, seed=41, bitdepth=8)
    col = OrderCollector(y, u, v)
    _lib.predict_stream_multi(hs, [[w[22], w[37]] for w in ws], 11, 256, 128, 1, col.read, col.write, window_frames=2)
    assert col.reads[0][0] == 0
    for (a, b, _), (c, _, _) in zip(col.reads, col.reads[1:]):
        assert c == a + b                       # ascending and contiguous
    assert sum(b for _, b, _ in col.reads) == 11
    assert [w[0] for w in col.windows] == list(range(0, 11, 2))
    assert col.threads == {threading.get_ident()} and col.devices == {torch.cuda.current_device()}


# ---- argument and consistency errors ----------------------------------------------------------------------------------
def test_multi_bad_arguments_call_nothing(handles):
    hs, ws = handles
    L = _lib.lib()
    calls = []
    rd = _lib.READ_CB(lambda *a: calls.append("read") or 0)
    wr = _lib.WRITE_CB(lambda *a: calls.append("write") or 0)

    def call(hlist, rows, n=None):
        n = len(hlist) if n is None else n
        arr = (ctypes.c_void_p * max(len(hlist), 1))(*[h.ptr if h is not None else None for h in hlist])
        flat = (ctypes.c_int * max(4 * len(rows) * len(rows[0]), 1))(*[x for by_qp in rows for r in by_qp for x in r])
        rc = L.pmp_predict_stream_multi(arr, n, len(rows[0]), flat, 2, 256, 128, 1, 0, 3, rd, wr, None, None)
        return rc, L.pmp_last_error().decode()

    good = [[w[32]] for w in ws]
    ok = ["read", "read", "write", "write"]          # 2 frames over 3 handles: two one-frame windows
    assert call(hs, good)[0] == 0 and calls == ok
    calls.clear()
    assert call(hs[:2], good[:2], n=0) == (-1, "bad argument: n_handles must be 1 to 16")
    assert call([hs[0]] * 17, [good[0]] * 17)[0] == -1 and "n_handles" in L.pmp_last_error().decode()
    rc, msg = call([hs[0], None, hs[2]], good)
    assert rc == -1 and "handles[1] is null" in msg
    rc, msg = call([hs[0], hs[1], hs[0]], good)
    assert rc == -1 and "handles[2] is handles[0]" in msg
    rc, msg = call(hs[:2], [[ws[0][32]], [ws[1][27]]])
    assert rc == -1 and "handles[1]" in msg and "weights of wsets[1][0][0]" in msg, msg
    no_chroma = ws[1][32][:2] + [-1, -1]
    rc, msg = call(hs[:2], [[ws[0][32]], [no_chroma]])
    assert rc == -1 and "handles[1]" in msg and "chroma of QP row 0 is skipped" in msg, msg
    rc, msg = call(hs[:2], [[ws[0][32]], [[ws[1][32][1], ws[1][32][0]] + ws[1][32][2:]]])      # Q and MSBD swapped
    assert rc == -1 and msg.startswith("handles[1]: ") and "net kind" in msg, msg
    hs[2].set_engine(_lib.ENGINE_TC, _lib.TC_BF16)
    try:
        rc, msg = call(hs, good)
        assert rc == -1 and "handles[2]" in msg and "tc_dtype 1" in msg, msg
    finally:
        hs[2].set_engine(_lib.ENGINE_TC, _lib.TC_FP16)
    hs[1].set_near_tol(2e-2)
    try:
        rc, msg = call(hs, good)
        assert rc == -1 and "handles[1]" in msg and "near_tol" in msg, msg
    finally:
        hs[1].set_near_tol(1e-2)
    assert calls == []
    assert call(hs, good)[0] == 0 and calls == ok


# ---- callback failures ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["read", "write"])
def test_multi_callback_failure_aborts(handles, which):
    hs, ws = handles
    y, u, v = synth.synth_yuv420(416, 240, 6, seed=38, bitdepth=8)
    # one-frame windows over two handles: read 3 is window 3, which handles[1] owns
    col = Collector(y, u, v, **{"fail_%s_at" % which: 3 if which == "read" else 2})
    with pytest.raises(_lib.PmpError, match=r"error -6: the %s callback returned %d" % (which, 3 if which == "read" else 5)):
        _lib.predict_stream_multi(hs[:2], [[w[22], w[37]] for w in ws[:2]], 6, 416, 240, 1, col.read, col.write,
                                  window_frames=1)
    if which == "read":
        assert [r[0] for r in col.reads] == [0, 1, 2, 3] and all(w[0] < 3 for w in col.windows)
    else:
        assert [w[0] for w in col.windows] == [0, 1, 2]
    # every handle is still usable and right
    got = hs[0].predict_host(ws[0][22], y, u, v)
    for h, w in zip(hs[:2], ws[:2]):
        again = Collector(y, u, v)
        h.predict_stream([w[22]], 6, 416, 240, 1, again.read, again.write, window_frames=4)
        for c in range(2):
            assert np.array_equal(np.concatenate(again.values[(0, c)]), got[c].reshape(-1))


def test_multi_python_exception_is_reraised(handles):
    hs, ws = handles
    y, u, v = synth.synth_yuv420(256, 128, 4, seed=39, bitdepth=8)
    col = Collector(y, u, v)

    def bad_read(f0, nf, yy, uu, vv):
        if f0 == 1:
            raise ValueError("no such frame")
        return col.read(f0, nf, yy, uu, vv)

    with pytest.raises(ValueError, match="no such frame") as e:
        _lib.predict_stream_multi(hs[:2], [[w[32]] for w in ws[:2]], 4, 256, 128, 1, bad_read, col.write, window_frames=1)
    assert isinstance(e.value.__context__, _lib.PmpError) and "-6" in str(e.value.__context__)
    assert [w[0] for w in col.windows] == []


# ---- saturation -------------------------------------------------------------------------------------------------------
def test_multi_stops_after_saturating_window(exported):
    sat = list(_saturating_luma_q().values())
    hs = [_lib.Handle(0) for _ in range(2)]
    try:
        rows = [[[h.weights_create("Luma_Q", sat), h.weights_load(str(exported / "Luma_BD_32.pmpw"))[1], -1, -1]]
                for h in hs]
        y, u, v = synth.synth_yuv420(256, 128, 5, seed=1, bitdepth=8)
        single = Collector(y, u, v)
        with pytest.raises(_lib.PmpError, match="error -4"):
            hs[0].predict_stream(rows[0], 5, 256, 128, 1, single.read, single.write, window_frames=1)
        col = Collector(y, u, v)
        rep = _lib.Report()
        with pytest.raises(_lib.PmpError) as e:
            _lib.predict_stream_multi(hs, rows, 5, 256, 128, 1, col.read, col.write, window_frames=1, report=rep)
        assert "error -4" in str(e.value) and "PMP_TC_BF16" in str(e.value)
        events = [w[2]["fp16_saturation_events"] for w in col.windows]
        assert events[-1] > 0 and all(n == 0 for n in events[:-1])       # written up to the first saturating window
        assert [w[0] for w in col.windows] == list(range(len(events)))
        assert [w[:2] for w in col.windows] == [w[:2] for w in single.windows]
        assert rep.fp16_saturation_events == sum(events) and rep.blocks == 8 * len(events)
    finally:
        for h in hs:
            h.close()


# ---- bounded staging --------------------------------------------------------------------------------------------------
def test_multi_memory_does_not_grow_with_frames(exported):
    hs = [_lib.Handle(0) for _ in range(2)]
    rows = [[w for w in _load_all(h, exported).values()] for h in hs]
    y, u, v = synth.synth_yuv420(416, 240, 40, seed=41, bitdepth=8)

    def run(f):
        col = Collector(y, u, v)
        _lib.predict_stream_multi(hs, rows, f, 416, 240, 1, col.read, lambda w: 0, window_frames=2)

    run(8)
    torch.cuda.synchronize()
    free8 = torch.cuda.mem_get_info()[0]
    run(40)
    torch.cuda.synchronize()
    free40 = torch.cuda.mem_get_info()[0]
    for h in hs:
        h.close()
    assert abs(free8 - free40) <= 8 << 20, (free8, free40)


# ---- the native tool's --devices ------------------------------------------------------------------------------------
def test_native_tool_stream_devices_matches_other_paths(exported, native_tool, tmp_path):
    y, u, v = synth.synth_yuv420(416, 240, 9, seed=21, bitdepth=8)
    seq = tmp_path / "seqD_416x240_8bit.yuv"
    _write_yuv(seq, y, u, v)
    args = ("--ssRatio", "2", "--binaryOut")
    runs = {"default": (), "stream": ("--stream", "--chunk", "20"),
            "devices": ("--stream", "--chunk", "20", "--devices", "0,0", "--timing"),
            "devices_default_window": ("--stream", "--devices", "0,0,0")}
    res = {k: _tool(native_tool, seq, 416, 240, 9, exported, tmp_path / k, *(args + extra)) for k, extra in runs.items()}
    for k, r in res.items():
        assert r.returncode == 0, (k, r.stderr)
        assert _report_line(r.stdout) == _report_line(res["default"].stdout)
    assert "pmp_predict_stream_multi" in res["devices"].stdout and "(5 frames, 5 windows, 2 handles)" in res["devices"].stdout
    files = sorted(os.listdir(tmp_path / "default"))
    assert len(files) == 16
    for k in runs:
        assert sorted(os.listdir(tmp_path / k)) == files, k
        for n in files:
            assert open(tmp_path / k / n, "rb").read() == open(tmp_path / "default" / n, "rb").read(), (k, n)
    # the golden files through two handles
    y, u, v = cases.pipeline_frames()
    seq = tmp_path / "pipe_192x128_10bit.yuv"
    _write_yuv(seq, y, u, v)
    r = _tool(native_tool, seq, 192, 128, cases.PIPE_F, exported, tmp_path / "pipe", "--bitDepth", "10", "--qps", "32",
              "--stream", "--devices", "0,0")
    assert r.returncode == 0, r.stderr
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    for comp in COMPS:
        want = open(os.path.join(golden, "pipeline_%s_QP32_PartitionMat.txt" % comp), "rb").read()
        assert open(tmp_path / "pipe" / ("pipe_192x128_10bit_%s_QP32_PartitionMat.txt" % comp), "rb").read() == want


# ---- distinct devices -------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more visible GPUs")
@pytest.mark.parametrize("devices", [(0, 1), (0, 1, 0, 1)])
def test_multi_distinct_devices(exported, devices):
    hs = [_lib.Handle(d) for d in devices]
    try:
        ws = [_load_all(h, exported) for h in hs]
        y, u, v = synth.synth_yuv420(832, 480, 9, seed=42)
        qps = (22, 37)
        ref = Collector(y, u, v)
        want_rep = hs[0].predict_stream([ws[0][q] for q in qps], 9, 832, 480, 2, ref.read, ref.write,
                                        window_frames=2).as_dict()
        for caller in (0, 1):
            with torch.cuda.device(caller):
                col = OrderCollector(y, u, v)
                rep = _lib.predict_stream_multi(hs, [[w[q] for q in qps] for w in ws], 9, 832, 480, 2, col.read,
                                                col.write, window_frames=2)
                assert torch.cuda.current_device() == caller
            assert col.devices == {caller} and col.threads == {threading.get_ident()}
            assert _joined(col) == _joined(ref) and rep.as_dict() == want_rep
    finally:
        for h in hs:
            h.close()
