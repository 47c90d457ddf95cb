"""Weight files: the reference's ``.pkl`` contract (Inference_QBD.py:28-46).

* files are legacy ``torch.save`` pickles of an OrderedDict (optionally wrapped in
  ``{"state_dict": ...}``), keys prefixed ``module.`` (saved from DataParallel), storages
  tagged CUDA -> always load with ``map_location='cpu'`` (the reference's own loader
  raises on a CPU-only host);
* ``load_pretrain_model`` keeps only keys present in the model with a matching shape and
  silently skips the rest.

Exported weight files (``.pmpw``, written by ``export_weights``) carry the same tensors in a flat, checksummed layout
that the C library reads without Python (``pmp_weights_load``).
"""
import os
import struct
from collections import OrderedDict

import numpy as np
import torch


def remove_prefix(state_dict, prefix):
    """Inference_QBD.py:28-30."""
    return {(k.split(prefix, 1)[-1] if k.startswith(prefix) else k): v for k, v in state_dict.items()}


def load_reference_pkl(path):
    """Read a reference ``.pkl`` into ``{name: cpu float tensor}`` with ``module.`` stripped."""
    src = torch.load(path, map_location="cpu", weights_only=False)
    if "state_dict" in src.keys():
        src = src["state_dict"]
    return remove_prefix(src, "module.")


def load_pretrain_model(current_model, pretrain_model):
    """Drop-in for Inference_QBD.load_pretrain_model (:33-46): shape-matched partial load."""
    source = load_reference_pkl(pretrain_model) if isinstance(pretrain_model, str) else \
        remove_prefix(pretrain_model, "module.")
    dest = current_model.state_dict()
    trained = {k: v for k, v in source.items() if k in dest and tuple(v.shape) == tuple(dest[k].shape)}
    dest.update(trained)
    current_model.load_state_dict(dest)
    return current_model


def reference_state_dicts(model_dir, comp, qp, missing_bd="error"):
    """(Q, MSBD) state dicts of one component and QP from the reference's file naming (Inference_QBD.py:219-220):
    <comp>_Q_<qp>.pkl, <comp>_BD_<qp>.pkl.  missing_bd="seeded" substitutes seeded random MSBD weights (seed
    1000 + qp, +500 for chroma) when the BD file is absent -- for benchmarking and tests only."""
    from . import synth
    sd_q = load_reference_pkl(os.path.join(model_dir, "%s_Q_%d.pkl" % (comp, qp)))
    bd_path = os.path.join(model_dir, "%s_BD_%d.pkl" % (comp, qp))
    if os.path.exists(bd_path):
        return sd_q, load_reference_pkl(bd_path)
    if missing_bd == "seeded":
        return sd_q, synth.seeded_state_dict(comp + "_MSBD", 1000 + qp + (0 if comp == "Luma" else 500))
    raise FileNotFoundError(bd_path)


# ---- exported weight files (.pmpw), read by pmp_weights_load ------------------------------------------------------
# Little-endian.  A 64-byte header: "PMPW0001", int32 net kind (enum pmp_net), int32 tensor count, int64 total floats,
# uint64 FNV-1a-64 of every byte after the header, zero padding.  Then per tensor: int32 name length, the name, int32 ndim,
# int32 dims[ndim]; zero padding to a multiple of 64 bytes; then the fp32 data of all tensors in record order.
PMPW_MAGIC = b"PMPW0001"
PMPW_HEADER = 64


def fnv1a64(data):
    h, prime, mask = 0xCBF29CE484222325, 0x100000001B3, 0xFFFFFFFFFFFFFFFF
    for b in data:
        h = ((h ^ b) * prime) & mask
    return h


def ordered_tensors(net, state_dict):
    """[(name, float32 array)] of `state_dict` (``module.`` prefix allowed) in param_spec(net) order; a missing tensor or
    a wrong shape raises."""
    from .netspec import param_spec
    sd = remove_prefix(dict(state_dict), "module.")
    out = []
    for name, shape in param_spec(net):
        if name not in sd:
            raise KeyError("%s: missing parameter %s" % (net, name))
        t = sd[name]
        a = np.asarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t)
        if tuple(a.shape) != tuple(shape):
            raise ValueError("%s: %s has shape %s, expected %s" % (net, name, tuple(a.shape), tuple(shape)))
        out.append((name, np.ascontiguousarray(a, dtype="<f4")))
    return out


def pmpw_bytes(net, state_dict):
    """The .pmpw image of `state_dict` for `net` ("Luma_Q", "Luma_MSBD", "Chroma_Q" or "Chroma_MSBD")."""
    from .netspec import NETS
    arrays = ordered_tensors(net, state_dict)
    recs = bytearray()
    for name, a in arrays:
        nb = name.encode()
        recs += struct.pack("<i", len(nb)) + nb + struct.pack("<i", a.ndim) + struct.pack("<%di" % a.ndim, *a.shape)
    recs += b"\0" * (-(PMPW_HEADER + len(recs)) % 64)
    body = bytes(recs) + b"".join(a.tobytes() for _, a in arrays)
    total = sum(a.size for _, a in arrays)
    head = PMPW_MAGIC + struct.pack("<iiqQ", NETS.index(net), len(arrays), total, fnv1a64(body))
    return head + b"\0" * (PMPW_HEADER - len(head)) + body


def write_pmpw(path, net, state_dict):
    data = pmpw_bytes(net, state_dict)
    with open(path, "wb") as fp:
        fp.write(data)
    return len(data)


def read_pmpw(path):
    """-> (net name, OrderedDict name -> float32 array).  Checks the magic, the records against param_spec, the size and
    the checksum."""
    from .netspec import NETS, param_spec
    with open(path, "rb") as fp:
        data = fp.read()
    if len(data) < PMPW_HEADER or data[:8] != PMPW_MAGIC:
        raise ValueError("%s: not a PMPW0001 file" % path)
    kind, n, total, csum = struct.unpack_from("<iiqQ", data, 8)
    if not 0 <= kind < len(NETS):
        raise ValueError("%s: unknown net kind %d" % (path, kind))
    net = NETS[kind]
    spec = param_spec(net)
    if n != len(spec):
        raise ValueError("%s: %d tensors, %s has %d" % (path, n, net, len(spec)))
    off, shapes = PMPW_HEADER, []
    for name, shape in spec:
        (ln,) = struct.unpack_from("<i", data, off)
        got = data[off + 4:off + 4 + ln].decode()
        (nd,) = struct.unpack_from("<i", data, off + 4 + ln)
        dims = struct.unpack_from("<%di" % nd, data, off + 8 + ln)
        if got != name or tuple(dims) != tuple(shape):
            raise ValueError("%s: record %s %s, expected %s %s" % (path, got, dims, name, tuple(shape)))
        shapes.append((name, dims))
        off += 8 + ln + 4 * nd
    off += -off % 64
    if total != sum(int(np.prod(s)) for _, s in shapes) or len(data) != off + 4 * total:
        raise ValueError("%s: size does not match the records" % path)
    if fnv1a64(data[PMPW_HEADER:]) != csum:
        raise ValueError("%s: checksum mismatch" % path)
    out = OrderedDict()
    for name, dims in shapes:
        k = int(np.prod(dims))
        out[name] = np.frombuffer(data, dtype="<f4", count=k, offset=off).reshape(dims).astype(np.float32)
        off += 4 * k
    return net, out
