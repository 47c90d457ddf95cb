"""The native tool's --devices option and predict_stream_multi's argument shape on the host: usage errors, the no-device
failure of the several-handle stream (tools/native/pmp_predict.cpp, pmp_vvc_tip2023_b200/_lib.py)."""
import os
import subprocess

import pytest
import torch

from pmp_vvc_tip2023_b200 import _lib, build

NO_GPU = not torch.cuda.is_available()


@pytest.fixture(scope="module")
def native_tool(tmp_path_factory):
    build.build()
    return build.build_native_tool(str(tmp_path_factory.mktemp("native") / "pmp_predict"))


def _run(tool, tmp_path, *extra):
    return subprocess.run([tool, "--input", str(tmp_path / "x.yuv"), "--width", "192", "--height", "128", "--frames", "2",
                           "--modelDir", str(tmp_path), "--outDir", str(tmp_path / "out")] + list(extra),
                          capture_output=True, text=True)


@pytest.mark.parametrize("extra, msg", [
    (("--devices", "0,1"), "needs --stream"),
    (("--devices", "0,0"), "needs --stream"),
    (("--stream", "--device", "0", "--devices", "0"), "exclude each other"),
    (("--stream", "--devices", "0", "--device", "1"), "exclude each other"),
    (("--stream", "--devices", ""), "device numbers"),
    (("--stream", "--devices", "0,,1"), "device numbers"),
    (("--stream", "--devices", "0,"), "device numbers"),
    (("--stream", "--devices", "0,x"), "device numbers"),
    (("--stream", "--devices", "-1"), "device numbers"),
    (("--stream", "--devices", ",".join(["0"] * 17)), "at most 16"),
])
def test_native_tool_devices_usage_errors(native_tool, tmp_path, extra, msg):
    r = _run(native_tool, tmp_path, *extra)
    assert r.returncode == 2 and msg in r.stderr and "[--device D | --devices D,D,...]" in r.stderr, r.stderr
    assert not os.path.exists(tmp_path / "out")


@pytest.mark.skipif(not NO_GPU, reason="checks the no-device failure mode")
def test_native_tool_stream_devices_fail_loudly_without_gpu(native_tool, tmp_path):
    r = _run(native_tool, tmp_path, "--stream", "--devices", "0,0")
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
    assert not os.path.exists(tmp_path / "out")


def test_predict_stream_multi_needs_one_row_list_per_handle():
    """The rows are checked in Python before the library is called: one list of the same QP count per handle."""
    def nothing(*_):
        return 0

    for rows in ([[[1, 2, 3, 4]]], [[[1, 2, 3, 4]], [[1, 2, 3, 4], [5, 6, 7, 8]]]):
        with pytest.raises(ValueError, match="one list of"):
            _lib.predict_stream_multi([1, 2], rows, 2, 256, 128, 1, nothing, nothing)
