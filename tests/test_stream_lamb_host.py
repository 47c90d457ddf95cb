"""The native tool's --lamb option and the lamb argument of the stream bindings on the host: usage errors, the no-device
failure of a threshold sweep (tools/native/pmp_predict.cpp, pmp_vvc_tip2023_b200/_lib.py)."""
import os
import subprocess

import pytest
import torch

from pmp_vvc_tip2023_b200 import _lib, build

NO_GPU = not torch.cuda.is_available()
DEFAULTS = "0.7,0.7,1.5,0.3,0.7"


@pytest.fixture(scope="module")
def native_tool(tmp_path_factory):
    build.build()
    return build.build_native_tool(str(tmp_path_factory.mktemp("native") / "pmp_predict"))


def _run(tool, tmp_path, *extra):
    return subprocess.run([tool, "--input", str(tmp_path / "x.yuv"), "--width", "192", "--height", "128", "--frames", "2",
                           "--modelDir", str(tmp_path), "--outDir", str(tmp_path / "out")] + list(extra),
                          capture_output=True, text=True)


@pytest.mark.parametrize("extra, msg", [
    (("--lamb", DEFAULTS), "--lamb needs --stream"),
    (("--lamb", DEFAULTS, "--devices", "0"), "--lamb needs --stream"),
    (("--stream", "--lamb", "0.7,0.7,1.5,0.3"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", DEFAULTS + ",0.1"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", "0.7,0.7,nan,0.3,0.7"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", "0.7,inf,1.5,0.3,0.7"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", "0.7,0.7,,0.3,0.7"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", "0.7,0.7,1.5x,0.3,0.7"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", DEFAULTS, "--lamb", "0.7,0.7,1.5,0.3"), "five comma-separated finite numbers"),
    (("--stream", "--lamb", DEFAULTS, "--lamb", DEFAULTS), "make 8 rows, at most 4"),       # 2 settings x 4 QPs
    (("--stream", "--qps", "22,32", "--lamb", DEFAULTS, "--lamb", DEFAULTS, "--lamb", DEFAULTS), "make 6 rows"),
])
def test_native_tool_lamb_usage_errors(native_tool, tmp_path, extra, msg):
    r = _run(native_tool, tmp_path, *extra)
    assert r.returncode == 2 and msg in r.stderr and "[--lamb l1,l2,l3,l4,l5 ...]" in r.stderr, r.stderr
    assert not os.path.exists(tmp_path / "out")


@pytest.mark.skipif(not NO_GPU, reason="checks the no-device failure mode")
@pytest.mark.parametrize("extra", [("--lamb", DEFAULTS), ("--lamb", DEFAULTS, "--lamb", "0.6,0.8,1.2,0.4,0.6"),
                                   ("--lamb", DEFAULTS, "--devices", "0,0")])
def test_native_tool_stream_lamb_fails_loudly_without_gpu(native_tool, tmp_path, extra):
    r = _run(native_tool, tmp_path, "--stream", "--qps", "32", *extra)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
    assert not os.path.exists(tmp_path / "out")


def test_stream_lamb_needs_one_five_tuple_per_row():
    """lamb is checked in Python before the library is called: one tuple of five thresholds per row."""
    def nothing(*_):
        return 0

    rows = [[1, 2, 3, 4], [1, 2, 3, 4]]
    for lamb in ([(0.7, 0.7, 1.5, 0.3, 0.7)], [(0.7, 0.7, 1.5, 0.3, 0.7)] * 3, [(0.7, 0.7, 1.5, 0.3)] * 2,
                 [(0.7, 0.7, 1.5, 0.3, 0.7, 0.1), (0.7, 0.7, 1.5, 0.3, 0.7)]):
        with pytest.raises(ValueError, match="one .* tuple per row"):
            _lib.predict_stream_multi([1], [rows], 2, 256, 128, 1, nothing, nothing, lamb=lamb)
