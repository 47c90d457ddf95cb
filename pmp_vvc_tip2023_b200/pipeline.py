"""Whole hot path on one GPU: planar YUV frames -> per-frame PartitionMat vectors (and files).

This is the call a user of the framework makes (bench.py's ``e2e`` leg times it): host frames are copied to the
device, cut into 68x68 / 3x34x34 blocks there (``pmp_cut_blocks``), pushed through the Q and MSBD nets, the QT
post-process, the map-to-partition decode and the frame assembly (``pmp_run_component``), and come back as int8
vectors in the order ``get_sequence_partition_for_VTM`` writes them (Map2Partition.py:401-412).
"""
import os

import numpy as np
import torch

from . import _lib, ops, synth, weights
from .netspec import QPS

COMPS = ("Luma", "Chroma")


class PartitionPredictor:
    def __init__(self, device=0, engine="tc", tc_dtype="fp16", chunk=1024, near_tol=1e-2):
        if not torch.cuda.is_available():
            raise _lib.PmpError("no CUDA device: pmp_vvc_tip2023_b200 has no CPU fallback")
        self.device = torch.device("cuda", int(device))
        # a private handle: engine, weight sets and activation arena belong to this predictor alone (two predictors on
        # one device -- e.g. a simt-vs-tc comparison -- do not disturb each other or the Model_QBD modules' default handle)
        self.handle = _lib.Handle(int(device))
        self.set_engine(engine, tc_dtype)
        self.handle.set_near_tol(near_tol)
        self.chunk = int(chunk)
        self._wsets = {}           # (comp, qp) -> (wset_q, wset_msbd)
        self._copy_stream = None   # device->host copies of finished components overlap the next component's kernels
        self.last_flags = {}       # (comp, qp) -> per-block decode flags of the last predict_frames call (device int32)
        self._pinned = {}          # key -> reusable pinned host staging buffer (to_host_pinned)

    def close(self):
        """Free the private handle (weight sets, arena).  Idempotent."""
        if self.handle is not None:
            self.handle.close()
            self.handle = None
            self._pinned = {}

    def __del__(self):
        try:
            self.close()
        except Exception:       # interpreter shutdown: the library may already be gone
            pass

    def set_engine(self, engine, tc_dtype="fp16"):
        eng = {"simt": _lib.ENGINE_SIMT, "tc": _lib.ENGINE_TC}[engine]
        self.handle.set_engine(eng, {"fp16": _lib.TC_FP16, "bf16": _lib.TC_BF16}[tc_dtype])
        self.engine = engine

    # ---- weights -------------------------------------------------------------------------------
    def load_state_dicts(self, comp, qp, sd_q, sd_bd):
        """sd_*: {reference parameter name: array/tensor} (``module.`` prefix allowed)."""
        out = []
        for kind, sd in (("Q", sd_q), ("MSBD", sd_bd)):
            net = "%s_%s" % (comp, kind)
            out.append(self.handle.weights_create(net, [a for _, a in weights.ordered_tensors(net, sd)]))
        old = self._wsets.pop((comp, qp), None)
        if old:
            for w in old:
                self.handle.weights_destroy(w)
        self._wsets[(comp, qp)] = tuple(out)

    def load_pkls(self, model_dir, comps=COMPS, qps=QPS, missing_bd="error"):
        """Reference file naming (Inference_QBD.py:219-220): <comp>_Q_<qp>.pkl, <comp>_BD_<qp>.pkl.
        missing_bd="seeded" substitutes seeded random MSBD weights (the trained BD files are not redistributable
        in this repo's mount) -- for benchmarking/tests only."""
        for comp in comps:
            for qp in qps:
                self.load_state_dicts(comp, qp, *weights.reference_state_dicts(model_dir, comp, qp, missing_bd))

    def load_seeded(self, comps=COMPS, qps=QPS, seed=0):
        for comp in comps:
            for qp in qps:
                self.load_state_dicts(comp, qp, synth.seeded_state_dict(comp + "_Q", seed + qp),
                                      synth.seeded_state_dict(comp + "_MSBD", seed + 1000 + qp))

    # ---- compute -------------------------------------------------------------------------------
    def to_device(self, a):
        if isinstance(a, torch.Tensor):
            return a.to(self.device, non_blocking=True)
        a = np.ascontiguousarray(a)
        if a.dtype == np.uint16:
            a = a.view(np.int16)              # torch has no uint16 arithmetic; the kernel reads raw 16-bit words
        return torch.from_numpy(a).to(self.device, non_blocking=True)

    def cut(self, y, u, v, comps=COMPS):
        y, u, v = self.to_device(y), self.to_device(u), self.to_device(v)
        return ops.cut_blocks(y, u, v, want_luma="Luma" in comps, want_chroma="Chroma" in comps, handle=self.handle)

    def predict_blocks(self, comp, qp, blocks, frames, bh, bw, want_maps=False):
        wq, wb = self._wsets[(comp, qp)]
        res = ops.run_component(wq, wb, comp == "Luma", blocks, frames, bh, bw, self.chunk, want_maps,
                                want_flags=not want_maps, handle=self.handle)
        self.last_flags[(comp, qp)] = res[-1]
        return res if want_maps else res[0]

    def counts(self):
        """Decode report of the last ``predict_frames`` call (synchronises): per (comp, qp) and in total, the number of
        64x64 blocks whose argmin was a float32 near-tie (``near_tie_blocks``) and whose maps hold a value within
        ``near_tol`` of a decision threshold (``near_threshold_blocks``) -- the blocks whose integer output may
        legitimately differ from a float32 evaluation of the reference; plus the fp16 range-guard events."""
        per = {"%s_QP%d" % k: ops.flag_counts(f) for k, f in self.last_flags.items()}
        tot = {key: sum(c[key] for c in per.values()) for key in ("blocks", "near_tie_blocks", "near_threshold_blocks",
                                                              "near_threshold_blocks_tight")}
        tot["fp16_saturation_events"] = self.handle.saturation_count()
        return {"total": tot, "per_component_qp": per}

    def predict_frames(self, y, u, v, qps=(32,), comps=COMPS, want_maps=False, host_out=None):
        """y [F,H,W], u/v [F,H/2,W/2] (uint8, or uint16/int16 holding 10-bit samples), host or device.
        Returns {(comp, qp): int8 CUDA tensor [F, per-frame values]} (or tuples with maps).

        host_out: optional {(comp, qp): pinned int8 host tensor [F, per-frame values]}; each finished component is then
        copied to the host on a side stream while the next one computes -- call ``synchronize()`` before reading them."""
        f, hgt, wid = y.shape
        bh, bw = hgt // 64, wid // 64
        lb, cb = self.cut(y, u, v, comps)
        out = {}
        for comp in comps:
            blocks = lb if comp == "Luma" else cb
            for qp in qps:
                res = self.predict_blocks(comp, qp, blocks, f, bh, bw, want_maps)
                out[(comp, qp)] = res
                if host_out is not None:
                    vec = res[0] if want_maps else res
                    if self._copy_stream is None:
                        self._copy_stream = torch.cuda.Stream(self.device)
                    done = torch.cuda.Event()
                    done.record(torch.cuda.current_stream(self.device))
                    with torch.cuda.stream(self._copy_stream):
                        self._copy_stream.wait_event(done)
                        host_out[(comp, qp)].copy_(vec, non_blocking=True)
                    vec.record_stream(self._copy_stream)
        return out

    def to_host_pinned(self, key, t, sync=True):
        """Device tensor -> a view of a reusable pinned host buffer kept per `key` (valid until the next call with that
        key).  Pageable ``.cpu()`` copies run at a few GB/s and dominate the gather of PartitionMat text at 4K."""
        n = t.numel()
        buf = self._pinned.get(key)
        if buf is None or buf.numel() < n or buf.dtype != t.dtype:
            buf = torch.empty(n + n // 16 + 1, dtype=t.dtype).pin_memory()
            self._pinned[key] = buf
        out = buf[:n]
        out.copy_(t.reshape(-1), non_blocking=True)
        if sync:
            torch.cuda.current_stream(self.device).synchronize()
        return out

    def synchronize(self):
        """Wait for the compute stream and for the host copies queued by ``predict_frames(host_out=...)``."""
        torch.cuda.current_stream(self.device).synchronize()
        if self._copy_stream is not None:
            self._copy_stream.synchronize()

    @staticmethod
    def partition_path(save_dir, seq_path_name, comp, qp):
        """Inference_QBD.py:237."""
        return os.path.join(save_dir, "%s_%s_QP%d_PartitionMat.txt" % (seq_path_name, comp, qp))

    def write_partition_file(self, values, path):
        text = ops.format_text(values, handle=self.handle)
        with open(path, "wb") as fp:
            fp.write(text.cpu().numpy().tobytes())
        return int(text.numel())
