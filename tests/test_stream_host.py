"""The native tool's --stream path on the host: argument errors and the no-device failure (tools/native/pmp_predict.cpp)."""
import os
import subprocess

import pytest
import torch

from pmp_vvc_tip2023_b200 import build

NO_GPU = not torch.cuda.is_available()


@pytest.fixture(scope="module")
def native_tool(tmp_path_factory):
    build.build()
    return build.build_native_tool(str(tmp_path_factory.mktemp("native") / "pmp_predict"))


def test_native_tool_stream_usage_error(native_tool, tmp_path):
    r = subprocess.run([native_tool, "--stream", "--input", str(tmp_path / "x.yuv"), "--width", "192", "--height", "128",
                        "--frames", "2", "--modelDir", str(tmp_path), "--outDir", str(tmp_path / "out"), "--bitDepth", "9"],
                       capture_output=True, text=True)
    assert r.returncode == 2 and "usage: pmp_predict" in r.stderr and "[--stream]" in r.stderr
    assert not os.path.exists(tmp_path / "out")


@pytest.mark.skipif(not NO_GPU, reason="checks the no-device failure mode")
def test_native_tool_stream_fails_loudly_without_gpu(native_tool, tmp_path):
    r = subprocess.run([native_tool, "--stream", "--input", str(tmp_path / "x.yuv"), "--width", "192", "--height", "128",
                        "--frames", "2", "--modelDir", str(tmp_path), "--outDir", str(tmp_path / "out")],
                       capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
    assert not os.path.exists(tmp_path / "out")
