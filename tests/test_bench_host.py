"""Host-side pieces of bench.py that need no GPU: the sha gate of `roofline.traffic`, the roofline peaks, the workload
description shared by both arms, the (QP, frame) shard arithmetic bench.py and Inference_QBD share, the output files of
--dump-outputs."""
import json
import os

import numpy as np
import torch

import bench
from pmp_vvc_tip2023_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_traffic_summary_matches_committed_kernel_sources():
    """The committed ncu DRAM summary was measured on exactly the kernel sources in the tree (bench.py reports
    `roofline.traffic` only then)."""
    traffic, src = bench.measured_traffic(4800)
    assert traffic is not None, src
    tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
    assert abs(traffic - tj["conv_tc_dram_bytes_per_launch_per_block"] * 4800) < 1.0
    # per launch and block the conv kernels move about the compulsory bytes (0.3 .. 1 MB), not multiples of them
    assert 0.3e6 < tj["conv_tc_dram_bytes_per_launch_per_block"] < 1.0e6


def test_stale_traffic_summary_is_refused(monkeypatch):
    monkeypatch.setattr(bench, "kernel_source_sha", lambda: "0" * 16)
    traffic, why = bench.measured_traffic(4800)
    assert traffic is None and "not reported" in why


def test_roofline_peaks_are_the_documented_measurements(monkeypatch, tmp_path):
    """Without a MEASURED_PEAKS.json the roofline is normalised by the peaks BASELINE.md records."""
    doc = open(os.path.join(ROOT, "BASELINE.md")).read()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    pk = bench.peaks()
    assert "BASELINE.md" in pk["src"]
    assert all(s in doc for s in ("HBM 6,446.6 GB/s", "1,660.1 TFLOP/s burst", "1,413.7 TFLOP/s sustained"))
    assert (pk["hbm_gbs"], pk["bf16_burst"], pk["bf16_sustained"]) == (6446.6, 1660.1, 1413.7)


def test_both_arms_carry_the_same_workload_config():
    a, b = bench.workload_config(), bench.workload_config("tc")
    assert a == b and a["units_per_step"] == 4800 and "configs[1]" in a["workload"]


def test_dump_outputs_writes_fixed_float32_samples(tmp_path):
    """--dump-outputs: one float32 .npy per (component, QP); outputs longer than the sample keep the values at the same
    seeded positions in every run; a full 1080p10 step stays under 64 MB."""
    # long outputs hold (position + 1) * qp, so every sampled value tells where it was taken
    res = {(c, q): (torch.arange(1000, dtype=torch.int32).reshape(2, 500) + 1) * q for c in ("Luma", "Chroma") for q in (22, 37)}
    res[("Luma", 27)] = torch.arange(-5, 5, dtype=torch.int8).reshape(2, 5)
    a, b = tmp_path / "a", tmp_path / "b"
    assert bench.dump_outputs(str(a), res, sample=300) == bench.dump_outputs(str(b), res, sample=300)
    assert sorted(os.listdir(a)) == sorted("%s_QP%d.npy" % k for k in res)
    positions = []
    for (c, q), t in res.items():
        x = np.load(a / ("%s_QP%d.npy" % (c, q)))
        assert x.dtype == np.float32 and np.array_equal(x, np.load(b / ("%s_QP%d.npy" % (c, q))))
        if q == 27:
            assert np.array_equal(x, np.arange(-5, 5))
        else:
            positions.append(x / q - 1)
    assert all(np.array_equal(p, positions[0]) for p in positions)
    assert positions[0].size == 300 and (np.diff(positions[0]) > 0).all() and positions[0][-1] < 1000
    cfg = bench.workload_config()
    outputs, per_output = 2 * len(cfg["qps"]), cfg["frames"] * 645120
    assert outputs * 4 * min(bench.DUMP_SAMPLE, per_output) <= 64 << 20


def test_bench_shards_tile_the_4k_sequence():
    for world in (1, 2, 4, 8):
        per_qp = {}
        for r in range(world):
            for qi, a, b in sharding.qp_frame_shards(30, 4, world, r):
                per_qp.setdefault(qi, []).append((a, b))
        assert sorted(per_qp) == [0, 1, 2, 3]
        assert all(s[0][0] == 0 and s[-1][1] == 30 for s in per_qp.values())
