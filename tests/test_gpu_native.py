"""Python-free deployment on the GPU: weight sets from exported .pmpw files (pmp_weights_load), the host-to-host entry point
pmp_predict_host against PartitionPredictor.predict_frames, and the native tool (tools/native/pmp_predict.cpp) against the
reference's files and the Python driver."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import nets_ref
from pmp_vvc_tip2023_b200 import _lib, build, export_weights, Inference_QBD, partition_io, synth, weights
from pmp_vvc_tip2023_b200.netspec import QPS, param_spec
from pmp_vvc_tip2023_b200.pipeline import PartitionPredictor
from tests import cases

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
MODELS = os.path.join(ROOT, "trained_models")
COMPS = ("Luma", "Chroma")


@pytest.fixture(scope="module")
def exported(tmp_path_factory):
    out = tmp_path_factory.mktemp("pmpw")
    export_weights.export(MODELS, str(out), missing_bd="seeded")
    return out


@pytest.fixture(scope="module")
def native_tool(tmp_path_factory):
    return build.build_native_tool(str(tmp_path_factory.mktemp("native") / "pmp_predict"))


@pytest.fixture(scope="module")
def predictors(exported):
    """(PartitionPredictor with the .pkl weights, Handle with the same weights from .pmpw: {qp: wsets[4]})."""
    pp = PartitionPredictor(0, engine="tc", chunk=4800)
    pp.load_pkls(MODELS, missing_bd="seeded")
    h = _lib.Handle(0)
    ws = {qp: [h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (c, t, qp))))[1] for c in COMPS for t in ("Q", "BD")]
          for qp in QPS}
    yield pp, h, ws
    pp.close()
    h.close()


def _forward(h, wq, wb, x, in_dtype):
    L = _lib.lib()
    n = x.shape[0]
    qt = torch.empty((n, 1, 8, 8), dtype=torch.float32, device="cuda")
    outs = [torch.empty((n, 2, 16, 16), dtype=torch.float32, device="cuda") for _ in range(3)]
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(L.pmp_forward_q(h.ptr, wq, ctypes.c_void_p(x.data_ptr()), in_dtype, n, ctypes.c_void_p(qt.data_ptr()), s))
    _lib.check(L.pmp_forward_msbd(h.ptr, wb, ctypes.c_void_p(x.data_ptr()), in_dtype, ctypes.c_void_p(qt.data_ptr()), n,
                                  *[ctypes.c_void_p(o.data_ptr()) for o in outs], s))
    torch.cuda.synchronize()
    return [qt.cpu()] + [o.cpu() for o in outs]


@pytest.mark.parametrize("comp", COMPS)
@pytest.mark.parametrize("qp", QPS)
def test_loaded_weights_equal_created_weights(exported, comp, qp):
    g = np.load(os.path.join(GOLDEN, "nets_golden.npz"))
    if comp == "Luma":
        x, dt = torch.from_numpy(g["by"]).unsqueeze(1).contiguous().cuda(), _lib.IN_U8
    else:
        x, dt = nets_ref.chroma_net_input(g["by"], g["bu"], g["bv"]).contiguous().cuda(), _lib.IN_F32
    h = _lib.Handle(0)
    sd_q, sd_bd = weights.reference_state_dicts(MODELS, comp, qp, "seeded")
    made = [h.weights_create(net, [sd[k] for k, _ in param_spec(net)]) for net, sd in ((comp + "_Q", sd_q),
                                                                                     (comp + "_MSBD", sd_bd))]
    loaded = []
    for tag, kind in (("Q", 0), ("BD", 1)):
        net, w = h.weights_load(str(exported / ("%s_%s_%d.pmpw" % (comp, tag, qp))))
        assert net == kind + (0 if comp == "Luma" else 2)
        loaded.append(w)
    a, b = _forward(h, made[0], made[1], x, dt), _forward(h, loaded[0], loaded[1], x, dt)
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    h.close()


def _damaged(data, how):
    d = bytearray(data)
    if how == "magic":
        d[:8] = b"PMPW0002"
    elif how == "net_kind":
        d[8:12] = (2).to_bytes(4, "little")               # a Chroma_Q header on Luma_Q records
    elif how == "checksum":
        d[-5] ^= 0x01
    elif how == "truncated":
        d = d[:-100]
    elif how == "renamed":
        i = d.index(b"conv_q2.weight")
        d[i:i + 7] = b"conv_qX"
    elif how == "dim":
        i = d.index(b"resblock_q2.left.0.weight") + len("resblock_q2.left.0.weight") + 4
        d[i:i + 4] = (63).to_bytes(4, "little")          # first dim 64 -> 63
    return bytes(d)


@pytest.mark.parametrize("how", ["magic", "net_kind", "checksum", "truncated", "renamed", "dim"])
def test_malformed_weight_files_are_refused(exported, tmp_path, how):
    good = str(exported / "Luma_Q_32.pmpw")
    bad = str(tmp_path / ("bad_%s.pmpw" % how))
    with open(bad, "wb") as fp:
        fp.write(_damaged(open(good, "rb").read(), how))
    h = _lib.Handle(0)
    _, w0 = h.weights_load(good)
    L = _lib.lib()
    net, ws = ctypes.c_int(-7), ctypes.c_int(-7)
    rc = L.pmp_weights_load(h.ptr, bad.encode(), ctypes.byref(net), ctypes.byref(ws))
    msg = L.pmp_last_error().decode()
    assert rc == -1 and bad in msg, (rc, msg)
    print(how, "->", msg)
    _, w1 = h.weights_load(good)
    assert w1 == w0 + 1                        # the refused file created no weight set
    h.close()


def _host_case(name):
    """(y, u, v, chunk) of one comparison case; y/u/v host numpy arrays."""
    if name == "pipe_192x128_10bit":
        y, u, v = cases.pipeline_frames()
        return y, u, v, 0
    if name == "416x240_8bit_5f":
        return synth.synth_yuv420(416, 240, 5, seed=11, bitdepth=8) + (0,)
    if name == "1080p_10bit_3f_windows":
        return synth.synth_yuv420(1920, 1080, 3, seed=12) + (700,)          # 480 blocks per frame: 3 one-frame windows
    if name == "832x480_8bit_1f":
        return synth.synth_yuv420(832, 480, 1, seed=13, bitdepth=8) + (0,)
    raise KeyError(name)


def _python_result(pp, y, u, v, qp, comps=COMPS):
    pp.last_flags = {}              # counts() below covers this call only
    res = pp.predict_frames(y, u, v, qps=(qp,), comps=comps)
    torch.cuda.synchronize()
    return {c: res[(c, qp)].cpu().numpy() for c in comps}, pp.counts()["total"]


@pytest.mark.parametrize("name", ["pipe_192x128_10bit", "416x240_8bit_5f", "1080p_10bit_3f_windows", "832x480_8bit_1f"])
def test_predict_host_equals_predict_frames(predictors, name):
    pp, h, ws = predictors
    y, u, v, chunk = _host_case(name)
    qp = 37 if "1080p" in name else 32
    want, counts = _python_result(pp, y, u, v, qp)
    rep = _lib.Report()
    got = h.predict_host(ws[qp], y, u, v, chunk=chunk, report=rep)
    for c, g in zip(COMPS, got):
        assert g.shape == want[c].shape and np.array_equal(g, want[c]), (name, c)
    # the decode report counts what PartitionPredictor.counts() counts for the same input
    r = rep.as_dict()
    assert r["fp16_saturation_events"] == 0
    for k in ("blocks", "near_tie_blocks", "near_threshold_blocks", "near_threshold_blocks_tight"):
        assert r[k] == counts[k], (k, r, counts)
    print(name, r)


def test_predict_host_pitched_and_pinned_inputs(predictors):
    """Rows wider than the frame (pitch > width * sample_bytes) go through the pinned staging; dense pinned tensors and
    pinned outputs are copied directly.  Same bytes either way."""
    pp, h, ws = predictors
    y, u, v = synth.synth_yuv420(416, 240, 4, seed=14)                    # 10-bit
    want, _ = _python_result(pp, y, u, v, 27)

    def padded(a, extra):
        big = np.full(a.shape[:2] + (a.shape[2] + extra,), 777, a.dtype)
        big[:, :, :a.shape[2]] = a
        return big[:, :, :a.shape[2]]

    py, pu, pv = padded(y, 24), padded(u, 40), padded(v, 40)
    assert py.strides[1] > y.shape[2] * 2 and pu.strides[1] == pv.strides[1]
    got = h.predict_host(ws[27], py, pu, pv, chunk=20)                     # 18 blocks per frame: 4 one-frame windows
    assert all(np.array_equal(g, want[c]) for c, g in zip(COMPS, got))
    pin = [torch.from_numpy(a.view(np.int16)).pin_memory() for a in (y, u, v)]
    outs = tuple(torch.full(want[c].shape, -9, dtype=torch.int8).pin_memory() for c in COMPS)
    got = h.predict_host(ws[27], *pin, chunk=40, outs=outs)
    assert all(np.array_equal(g.numpy(), want[c]) for c, g in zip(COMPS, got))


@pytest.mark.parametrize("comp", COMPS)
def test_predict_host_one_component(predictors, comp):
    pp, h, ws = predictors
    y, u, v = synth.synth_yuv420(416, 240, 2, seed=15, bitdepth=8)
    want, counts = _python_result(pp, y, u, v, 22, comps=(comp,))
    sel = list(ws[22])
    skip = 2 if comp == "Luma" else 0
    sel[skip:skip + 2] = [-1, -1]
    rep = _lib.Report()
    got = h.predict_host(sel, y, None if comp == "Luma" else u, None if comp == "Luma" else v, report=rep)
    keep = 0 if comp == "Luma" else 1
    assert got[1 - keep] is None and np.array_equal(got[keep], want[comp])
    assert rep.blocks == counts["blocks"] == 2 * 3 * 6


def test_predict_host_small_frames_and_bad_arguments(predictors):
    _, h, ws = predictors
    y, u, v = synth.synth_yuv420(64, 62, 1, seed=1, bitdepth=8)
    out = np.full(8, 5, np.int8)
    rep = _lib.Report()
    rep.blocks = 99
    h.predict_host(ws[32], y, u, v, outs=(out, out), report=rep)          # height < 64: zero blocks, nothing written
    assert (out == 5).all() and rep.blocks == 0
    y, u, v = synth.synth_yuv420(128, 64, 1, seed=1, bitdepth=8)
    with pytest.raises(_lib.PmpError, match="net kind"):
        h.predict_host([ws[32][1], ws[32][0], ws[32][2], ws[32][3]], y, u, v)


def test_predict_host_reports_fp16_saturation(exported):
    """The weights of test_fp16_saturation_is_reported (one conv scaled by 2000) make activations leave the fp16 range:
    the call refuses with PMP_ERR_STATE and counts the events; the handle's sticky counter keeps its total."""
    h = _lib.Handle(0)
    sdq = synth.seeded_state_dict("Luma_Q", 3)
    big = [v * 2000.0 if k.startswith("resblock_q1.left.0") else v for k, v in sdq.items()]
    wq = h.weights_create("Luma_Q", big)
    _, wb = h.weights_load(str(exported / "Luma_BD_32.pmpw"))
    y, u, v = synth.synth_yuv420(256, 128, 2, seed=1, bitdepth=8)
    before = h.saturation_count()
    rep = _lib.Report()
    with pytest.raises(_lib.PmpError) as e:
        h.predict_host([wq, wb, -1, -1], y, None, None, report=rep)
    assert "error -4" in str(e.value) and "PMP_TC_BF16" in str(e.value)
    assert rep.fp16_saturation_events > 0 and rep.blocks == 16
    assert h.saturation_count() == before + rep.fp16_saturation_events
    h.close()


def _write_yuv(path, y, u, v):
    with open(path, "wb") as fp:
        for f in range(y.shape[0]):
            fp.write(y[f].tobytes()); fp.write(u[f].tobytes()); fp.write(v[f].tobytes())


def test_native_tool_matches_reference_files(exported, native_tool, tmp_path):
    y, u, v = cases.pipeline_frames()
    seq = tmp_path / "pipe_192x128_10bit.yuv"
    _write_yuv(seq, y, u, v)
    out = tmp_path / "out"
    r = subprocess.run([native_tool, "--input", str(seq), "--width", "192", "--height", "128", "--frames", str(cases.PIPE_F),
                        "--bitDepth", "10", "--ssRatio", "1", "--qps", "32", "--modelDir", str(exported), "--outDir", str(out),
                        "--binaryOut", "--timing"], capture_output=True, text=True)
    print(r.stdout, r.stderr)
    assert r.returncode == 0 and "Decode report: 24 block-QPs" in r.stdout and "pmp_predict_host" in r.stdout
    for comp in COMPS:
        got = open(out / ("pipe_192x128_10bit_%s_QP32_PartitionMat.txt" % comp), "rb").read()
        want = os.path.join(GOLDEN, "pipeline_%s_QP32_PartitionMat.txt" % comp)
        assert got == open(want, "rb").read()
        vals, rows, cols = partition_io.read_partition_bin(str(out / ("pipe_192x128_10bit_%s_QP32_PartitionMat.bin" % comp)))
        assert (rows, cols) == (32, 48)
        assert np.array_equal(vals, partition_io.text_to_values(want, cases.PIPE_H, cases.PIPE_W))


def test_native_tool_matches_python_driver(exported, native_tool, tmp_path):
    y, u, v = synth.synth_yuv420(416, 240, 9, seed=21, bitdepth=8)
    inp = tmp_path / "in"
    inp.mkdir()
    name = "seqD_416x240_8bit.yuv"
    _write_yuv(inp / name, y, u, v)
    (tmp_path / "seqs.txt").write_text("seqD,%s,416,240,9,4\n#end!!!!\n" % name)
    args = Inference_QBD.build_parser().parse_args([
        "--jobID", "j", "--inputDir", str(inp), "--outDir", str(tmp_path / "py"), "--batchSize", "200", "--seqNum", "1",
        "--seqInfo", str(tmp_path / "seqs.txt"), "--cfgDir", str(tmp_path / "nocfg"), "--modelDir", MODELS, "--ssRatio", "4",
        "--missingBD", "seeded", "--gpus", "1", "--binaryOut"])
    Inference_QBD.inference_VVC_seqs(args)
    py_dir = tmp_path / "py" / "j" / "PartitionMat"
    cmd = [native_tool, "--input", str(inp / name), "--width", "416", "--height", "240", "--frames", "9", "--ssRatio", "4",
           "--modelDir", str(exported), "--outDir", str(tmp_path / "native")]
    r = subprocess.run(cmd + ["--binaryOut"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    files = sorted(n for n in os.listdir(py_dir))
    assert len(files) == 16
    for n in files:
        assert open(py_dir / n, "rb").read() == open(tmp_path / "native" / n, "rb").read(), n
    # without --binaryOut a stale .bin beside the new .txt is removed
    r = subprocess.run(cmd + ["--qps", "27"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    left = sorted(os.listdir(tmp_path / "native"))
    assert "seqD_416x240_8bit_Luma_QP27_PartitionMat.bin" not in left and "seqD_416x240_8bit_Luma_QP22_PartitionMat.bin" in left
    assert len(left) == 14
