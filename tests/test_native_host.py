"""Python-free deployment, host side: the .pmpw weight export (export_weights.py, weights.pmpw_bytes / read_pmpw) and the
native PartitionMat tool (tools/native/pmp_predict.cpp), which builds with g++ against the C header alone."""
import os
import struct
import subprocess

import numpy as np
import pytest
import torch

from pmp_vvc_tip2023_b200 import build, export_weights, netspec, synth, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODELS = os.path.join(ROOT, "trained_models")
NO_GPU = not torch.cuda.is_available()


@pytest.fixture(scope="module")
def exported(tmp_path_factory):
    out = tmp_path_factory.mktemp("pmpw")
    export_weights.main(["--modelDir", MODELS, "--outDir", str(out), "--missingBD", "seeded"])
    return out


def test_export_matches_spec_and_sources(exported):
    names = sorted(os.listdir(exported))
    assert names == sorted("%s_%s_%d.pmpw" % (c, t, q) for c in ("Luma", "Chroma") for t in ("Q", "BD") for q in netspec.QPS)
    for comp in ("Luma", "Chroma"):
        for qp in netspec.QPS:
            sd_q = weights.load_reference_pkl(os.path.join(MODELS, "%s_Q_%d.pkl" % (comp, qp)))
            sd_bd = synth.seeded_state_dict(comp + "_MSBD", 1000 + qp + (0 if comp == "Luma" else 500))
            for tag, net, want in (("Q", comp + "_Q", sd_q), ("BD", comp + "_MSBD", sd_bd)):
                path = str(exported / ("%s_%s_%d.pmpw" % (comp, tag, qp)))
                data = open(path, "rb").read()
                spec = netspec.param_spec(net)
                # header: magic, net kind, tensor count, total floats; then the records in param_spec order
                assert data[:8] == b"PMPW0001"
                kind, n, total = struct.unpack_from("<iiq", data, 8)
                assert (kind, n, total) == (netspec.NETS.index(net), len(spec), netspec.param_count(net))
                assert data[32:64] == b"\0" * 32
                off = 64
                for name, shape in spec:
                    (ln,) = struct.unpack_from("<i", data, off)
                    assert data[off + 4:off + 4 + ln] == name.encode()
                    (nd,) = struct.unpack_from("<i", data, off + 4 + ln)
                    assert struct.unpack_from("<%di" % nd, data, off + 8 + ln) == tuple(shape)
                    off += 8 + ln + 4 * nd
                off += -off % 64
                assert len(data) == off + 4 * total
                got_net, got = weights.read_pmpw(path)
                assert got_net == net and list(got) == [k for k, _ in spec]
                for k, a in got.items():
                    w = want[k]
                    w = w.numpy() if hasattr(w, "numpy") else w
                    assert a.dtype == np.float32 and np.array_equal(a, w), (path, k)


def test_export_is_deterministic(exported, tmp_path):
    export_weights.export(MODELS, str(tmp_path), missing_bd="seeded")
    for name in os.listdir(exported):
        assert open(exported / name, "rb").read() == open(tmp_path / name, "rb").read(), name


def test_export_without_bd_files_needs_seeded(tmp_path):
    with pytest.raises(FileNotFoundError):
        export_weights.export(MODELS, str(tmp_path), comps=("Luma",), qps=(32,))


@pytest.mark.parametrize("damage", ["missing", "reshaped"])
def test_export_refuses_incomplete_pkl(tmp_path, damage):
    raw = torch.load(os.path.join(MODELS, "Luma_Q_22.pkl"), map_location="cpu", weights_only=False)
    key = "module.resblock_q3.left.2.weight"
    assert key in raw
    if damage == "missing":
        del raw[key]
    else:
        raw[key] = raw[key].reshape(raw[key].shape[0], -1)
    models = tmp_path / "models"
    models.mkdir()
    torch.save(raw, str(models / "Luma_Q_22.pkl"))
    with pytest.raises(KeyError if damage == "missing" else ValueError, match="resblock_q3.left.2.weight"):
        export_weights.export(str(models), str(tmp_path / "out"), missing_bd="seeded", comps=("Luma",), qps=(22,))


def test_read_pmpw_rejects_a_flipped_byte(exported, tmp_path):
    data = bytearray(open(exported / "Chroma_Q_37.pmpw", "rb").read())
    data[-3] ^= 0x10
    bad = tmp_path / "bad.pmpw"
    bad.write_bytes(bytes(data))
    with pytest.raises(ValueError, match="checksum"):
        weights.read_pmpw(str(bad))


@pytest.fixture(scope="module")
def native_tool(tmp_path_factory):
    build.build()
    return build.build_native_tool(str(tmp_path_factory.mktemp("native") / "pmp_predict"))


def test_native_tool_compiles(native_tool):
    assert os.access(native_tool, os.X_OK)
    r = subprocess.run([native_tool, "--width", "64"], capture_output=True, text=True)
    assert r.returncode == 2 and "usage: pmp_predict" in r.stderr


@pytest.mark.skipif(not NO_GPU, reason="checks the no-device failure mode")
def test_native_tool_fails_loudly_without_gpu(native_tool, tmp_path):
    r = subprocess.run([native_tool, "--input", str(tmp_path / "x.yuv"), "--width", "192", "--height", "128", "--frames", "2",
                        "--modelDir", str(tmp_path), "--outDir", str(tmp_path / "out")], capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
    assert not os.path.exists(tmp_path / "out")
