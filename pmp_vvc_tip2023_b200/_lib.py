"""ctypes binding of libpmp_b200.so (include/pmp_b200.h).  No CPU fallback: every entry point
raises if the library is missing or no B200 is visible."""
import ctypes
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
# PMP_B200_LIB: file name of another build of the same library inside this directory (kernel A/B runs in one GPU call)
LIB_PATH = os.path.join(HERE, os.path.basename(os.environ.get("PMP_B200_LIB", "libpmp_b200.so")))

NET_LUMA_Q, NET_LUMA_MSBD, NET_CHROMA_Q, NET_CHROMA_MSBD = 0, 1, 2, 3
NET_IDS = {"Luma_Q": 0, "Luma_MSBD": 1, "Chroma_Q": 2, "Chroma_MSBD": 3}
ENGINE_SIMT, ENGINE_TC = 0, 1
TC_FP16, TC_BF16 = 0, 1
IN_U8, IN_F32 = 0, 1

c_void_p, c_int, c_int64, c_char_p = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_char_p
_P = ctypes.POINTER

class Report(ctypes.Structure):
    """struct pmp_report (pmp_predict_host)."""
    _fields_ = [(k, ctypes.c_longlong) for k in ("blocks", "near_tie_blocks", "near_threshold_blocks",
                                                 "near_threshold_blocks_tight", "fp16_saturation_events")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class Window(ctypes.Structure):
    """struct pmp_window (pmp_predict_stream): one window's results, [qp index][0 luma, 1 chroma]."""
    _fields_ = [("first_frame", c_int), ("frames", c_int), ("n_qps", c_int),
                ("values", (c_void_p * 2) * 4), ("n_values", (c_int64 * 2) * 4),
                ("text", (c_void_p * 2) * 4), ("text_bytes", (c_int64 * 2) * 4), ("report", Report)]


OUT_VALUES, OUT_TEXT = 1, 2
READ_CB = ctypes.CFUNCTYPE(c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p)
WRITE_CB = ctypes.CFUNCTYPE(c_int, c_void_p, _P(Window))

# name -> (restype, argtypes); kept in one table so tests can check the ABI against the header
SIGNATURES = {
    "pmp_version": (c_int, []),
    "pmp_last_error": (c_char_p, []),
    "pmp_create": (c_int, [c_int, _P(c_void_p)]),
    "pmp_destroy": (None, [c_void_p]),
    "pmp_set_engine": (c_int, [c_void_p, c_int, c_int]),
    "pmp_get_engine": (c_int, [c_void_p]),
    "pmp_set_near_tol": (c_int, [c_void_p, ctypes.c_float]),
    "pmp_saturation_count": (c_int, [c_void_p, _P(ctypes.c_longlong), c_int]),
    "pmp_launch_count": (ctypes.c_longlong, [c_void_p]),
    "pmp_profile": (c_int, [c_void_p, c_int]),
    "pmp_profile_read": (c_int, [c_void_p, c_int, c_char_p, c_int, _P(ctypes.c_double), _P(ctypes.c_longlong),
                                 _P(ctypes.c_double), _P(ctypes.c_double)]),
    "pmp_weights_create": (c_int, [c_void_p, c_int, _P(c_void_p), _P(c_int64), c_int, _P(c_int)]),
    "pmp_weights_destroy": (c_int, [c_void_p, c_int]),
    "pmp_weights_load": (c_int, [c_void_p, c_char_p, _P(c_int), _P(c_int)]),
    "pmp_predict_host": (c_int, [c_void_p, _P(c_int), c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int, c_int,
                                 c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "pmp_forward_q": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "pmp_forward_msbd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "pmp_predict_maps": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "pmp_qt_postprocess": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "pmp_map2partition": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p]),
    "pmp_map2partition_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, _P(ctypes.c_double), c_void_p,
                                     ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmp_assemble_frames": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                    c_void_p]),
    "pmp_frame_values": (c_int64, [c_int, c_int]),
    "pmp_format_text": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, _P(c_int64), c_void_p]),
    "pmp_format_texts": (c_int, [c_void_p, c_int, _P(c_void_p), _P(c_int64), _P(c_void_p), c_void_p, c_void_p]),
    "pmp_predict_stream": (c_int, [c_void_p, c_int, _P(c_int), c_int, c_int, c_int, c_int, c_int, c_int, READ_CB, WRITE_CB,
                                   c_void_p, _P(Report)]),
    "pmp_predict_stream_multi": (c_int, [_P(c_void_p), c_int, c_int, _P(c_int), c_int, c_int, c_int, c_int, c_int, c_int,
                                         READ_CB, WRITE_CB, c_void_p, _P(Report)]),
    "pmp_predict_stream_ex": (c_int, [_P(c_void_p), c_int, c_int, _P(c_int), _P(ctypes.c_double), c_int, c_int, c_int, c_int,
                                      c_int, c_int, READ_CB, WRITE_CB, c_void_p, _P(Report)]),
    "pmp_cut_blocks": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                               c_void_p]),
    "pmp_run_component": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pmp_selftest_conv": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, _P(ctypes.c_double),
                                  _P(ctypes.c_double), _P(ctypes.c_double), _P(ctypes.c_double)]),
    "pmp_debug_conv": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                               c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "pmp_debug_stem": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "pmp_debug_tc_stalls": (c_int, [_P(ctypes.c_uint64), c_int]),
    "pmp_block_stats": (c_int, [c_void_p, _P(ctypes.c_longlong), _P(ctypes.c_longlong), c_int]),
    "pmp_debug_block_groups": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, _P(c_int), c_void_p]),
}

_lib = None
_lock = threading.Lock()


class PmpError(RuntimeError):
    pass


def lib():
    """Load libpmp_b200.so (raises if it has not been built: there is no fallback path)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise PmpError("libpmp_b200.so is not built (%s); run `python -m pmp_vvc_tip2023_b200.build` "
                               "-- there is no CPU/PyTorch fallback" % LIB_PATH)
            L = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(L, name)
                fn.restype = res
                fn.argtypes = args
            _lib = L
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().pmp_last_error()
        raise PmpError("libpmp_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))


class Handle:
    """A pmp_handle (engine selection, weight sets, activation arena).  ``Handle.get(device)`` is the per-(process, device)
    default used by the Model_QBD modules and the module-level ops; a PartitionPredictor owns a private one, so that its
    engine choice and arena are its own.  Not thread-safe; one stream at a time per handle."""
    _cache = {}

    def __init__(self, device=0):
        self.device = int(device)
        self._h = c_void_p()
        check(lib().pmp_create(self.device, ctypes.byref(self._h)))
        self._wsets = []

    @classmethod
    def get(cls, device=0):
        device = int(device)
        if device not in cls._cache:
            cls._cache[device] = cls(device)
        return cls._cache[device]

    @property
    def ptr(self):
        return self._h

    def close(self):
        if self._h:
            lib().pmp_destroy(self._h)
            self._h = c_void_p()
        if Handle._cache.get(self.device) is self:
            Handle._cache.pop(self.device, None)

    # ---- engine / counters ------------------------------------------------------------------
    def set_engine(self, engine, tc_dtype=TC_FP16):
        check(lib().pmp_set_engine(self._h, engine, tc_dtype))

    def engine(self):
        return lib().pmp_get_engine(self._h)

    def set_near_tol(self, tol):
        check(lib().pmp_set_near_tol(self._h, float(tol)))

    def saturation_count(self, reset=False):
        """fp16 range-guard events of the TC conv epilogues (non-zero => results clamped: use tc_dtype='bf16')."""
        n = ctypes.c_longlong()
        check(lib().pmp_saturation_count(self._h, ctypes.byref(n), 1 if reset else 0))
        return int(n.value)

    def launch_count(self):
        return int(lib().pmp_launch_count(self._h))

    def block_stats(self, reset=False):
        """(blocks, computed): the blocks of the window pipeline's net passes on this handle and the distinct blocks the
        nets ran on (repeated blocks in a window are computed once), since creation or the last reset."""
        b, c = ctypes.c_longlong(), ctypes.c_longlong()
        check(lib().pmp_block_stats(self._h, ctypes.byref(b), ctypes.byref(c), 1 if reset else 0))
        return int(b.value), int(c.value)

    def profile(self, mode):
        check(lib().pmp_profile(self._h, mode))

    def profile_read(self):
        out = {}
        name = ctypes.create_string_buffer(64)
        for i in range(16):
            ms, n, fl, by = ctypes.c_double(), ctypes.c_longlong(), ctypes.c_double(), ctypes.c_double()
            rc = lib().pmp_profile_read(self._h, i, name, 64, ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl),
                                        ctypes.byref(by))
            if rc != 0:
                break
            out[name.value.decode()] = {"ms": ms.value, "launches": n.value, "flops": fl.value, "bytes": by.value}
        return out

    # ---- weights ----------------------------------------------------------------------------
    def weights_create(self, net, tensors):
        """tensors: list of contiguous float32 numpy arrays / CPU torch tensors in state_dict order."""
        import numpy as np
        arrs = [np.ascontiguousarray(t.detach().cpu().numpy() if hasattr(t, "detach") else t, dtype=np.float32)
                for t in tensors]
        n = len(arrs)
        ptrs = (c_void_p * n)(*[a.ctypes.data for a in arrs])
        numel = (c_int64 * n)(*[a.size for a in arrs])
        wset = c_int()
        net_id = NET_IDS[net] if isinstance(net, str) else int(net)
        check(lib().pmp_weights_create(self._h, net_id, ptrs, numel, n, ctypes.byref(wset)))
        return wset.value

    def weights_destroy(self, wset):
        check(lib().pmp_weights_destroy(self._h, wset))

    def weights_load(self, path):
        """An exported .pmpw file (export_weights.py) -> (net kind, weight-set id)."""
        net, wset = c_int(), c_int()
        check(lib().pmp_weights_load(self._h, os.fsencode(path), ctypes.byref(net), ctypes.byref(wset)))
        return net.value, wset.value

    # ---- host path ----------------------------------------------------------------------------
    def predict_host(self, wsets, y, u, v, chunk=0, outs=(None, None), report=None):
        """pmp_predict_host.  wsets: (luma Q, luma MSBD, chroma Q, chroma MSBD), -1, -1 skips a component.
        y [F,H,W], u/v [F,H/2,W/2]: host numpy arrays (uint8, or uint16 holding 10-bit samples) or CPU tensors; rows may
        be padded (a view of the first W columns of wider rows).  outs: (luma, chroma) host buffers of
        F * pmp_frame_values(H/64, W/64) int8 (numpy arrays or pinned tensors), None = allocate.  Returns the two
        outputs as int8 [F, per] (None for a skipped component); `report` (a Report) receives the decode report."""
        import numpy as np

        y, u, v = (a.numpy() if hasattr(a, "data_ptr") else a for a in (y, u, v))

        def plane(a):
            if a is None:
                return None, 0
            assert a.ndim == 3 and a.strides[2] == a.itemsize and a.strides[0] == a.shape[1] * a.strides[1]
            return c_void_p(a.ctypes.data), a.strides[1]

        f, hgt, wid = y.shape
        per = int(lib().pmp_frame_values(hgt // 64, wid // 64))
        res = []
        for i, o in enumerate(outs):
            if wsets[2 * i] == -1 and wsets[2 * i + 1] == -1:
                res.append(None)
            else:
                res.append(np.empty((f, per), np.int8) if o is None else o)
        ptr = [None if o is None else c_void_p(o.data_ptr() if hasattr(o, "data_ptr") else o.ctypes.data) for o in res]
        (py, sy), (pu, sc), (pv, _) = plane(y), plane(u), plane(v)
        report = Report() if report is None else report
        check(lib().pmp_predict_host(self._h, (c_int * 4)(*wsets), py, pu, pv, y.itemsize, sy, sc, f, wid, hgt, int(chunk),
                                     ptr[0], ptr[1], ctypes.byref(report)))
        return res

    def predict_stream(self, wsets_by_qp, frames, width, height, sample_bytes, read, write, window_frames=0,
                       outputs=OUT_VALUES | OUT_TEXT, report=None, lamb=None):
        """pmp_predict_stream.  wsets_by_qp: one (luma Q, luma MSBD, chroma Q, chroma MSBD) row per QP (1 to 4 rows).
        read(first_frame, frames, y, u, v) fills numpy views of the library's page-locked planes: y [frames, H, W],
        u/v [frames, H/2, W/2] (None when no QP runs chroma), uint8 or uint16 after sample_bytes.
        write(w) receives a StreamWindow per window, in frame order; its arrays are views valid only during the call.
        A non-zero return of a callback aborts the call (PmpError, error -6); an exception raised in a callback aborts
        it too and is re-raised here, chained to that error.  Returns the Report summed over the windows written.
        lamb: None, or one (lamb1..lamb5) decode-threshold tuple per row (pmp_predict_stream_ex on this handle); rows with
        equal weight sets share their net pass."""
        if lamb is not None:
            return predict_stream_multi([self], [wsets_by_qp], frames, width, height, sample_bytes, read, write,
                                        window_frames, outputs, report, lamb)
        rows = [list(r) for r in wsets_by_qp]
        flat = (c_int * (4 * max(len(rows), 1)))(*[w for r in rows for w in r])
        return _stream_call(lambda rd, wr, rep: lib().pmp_predict_stream(
            self._h, len(rows), flat, int(frames), int(width), int(height), int(sample_bytes), int(window_frames),
            int(outputs), rd, wr, None, rep), width, height, sample_bytes, read, write, report)


def predict_stream_multi(handles, wsets_by_handle, frames, width, height, sample_bytes, read, write, window_frames=0,
                         outputs=OUT_VALUES | OUT_TEXT, report=None, lamb=None):
    """pmp_predict_stream_multi: Handle.predict_stream over several handles (1 to 16, on one or several devices), window
    k on handles[k % len(handles)].  wsets_by_handle[i]: handles[i]'s rows, one (luma Q, luma MSBD, chroma Q,
    chroma MSBD) per QP, the same QPs and weights on every handle.  The callbacks, errors and result are those of
    Handle.predict_stream; the calling thread's current device is current inside the callbacks and after the call.
    lamb: None, or one (lamb1..lamb5) decode-threshold tuple per row (pmp_predict_stream_ex): row r's results are
    decoded with lamb[r]; a wrong length raises ValueError before the library is called."""
    nh = len(handles)
    rows = [[list(r) for r in by_qp] for by_qp in wsets_by_handle]
    nq = len(rows[0]) if rows else 0
    if len(rows) != nh or any(len(r) != nq for r in rows):
        raise ValueError("wsets_by_handle needs one list of %d QP rows per handle" % nq)
    flat = (c_int * (4 * max(nh * nq, 1)))(*[w for by_qp in rows for r in by_qp for w in r])
    hs = (c_void_p * max(nh, 1))(*[h.ptr if isinstance(h, Handle) else h for h in handles])
    if lamb is None:
        return _stream_call(lambda rd, wr, rep: lib().pmp_predict_stream_multi(
            hs, nh, nq, flat, int(frames), int(width), int(height), int(sample_bytes), int(window_frames), int(outputs),
            rd, wr, None, rep), width, height, sample_bytes, read, write, report)
    lamb = [tuple(t) for t in lamb]
    if len(lamb) != nq or any(len(t) != 5 for t in lamb):
        raise ValueError("lamb needs one (lamb1, lamb2, lamb3, lamb4, lamb5) tuple per row: %d rows" % nq)
    lam = (ctypes.c_double * (5 * max(nq, 1)))(*[float(x) for t in lamb for x in t])
    return _stream_call(lambda rd, wr, rep: lib().pmp_predict_stream_ex(
        hs, nh, nq, flat, lam, int(frames), int(width), int(height), int(sample_bytes), int(window_frames),
        int(outputs), rd, wr, None, rep), width, height, sample_bytes, read, write, report)


def _stream_call(call, width, height, sample_bytes, read, write, report):
    """Runs call(read_cb, write_cb, report_ptr) -> status with the Python callbacks of predict_stream wrapped: numpy views
    of the planes and StreamWindows in, a callback's exception re-raised here chained to the -6 it caused."""
    import numpy as np

    dt = np.uint8 if sample_bytes == 1 else np.uint16
    raised = []

    def view(ptr, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if not ptr:
            return None
        if n == 0:
            return np.empty(shape, dtype)
        return np.frombuffer((ctypes.c_char * n).from_address(ptr), dtype).reshape(shape)

    def on_read(_user, f0, nf, y, u, v):
        try:
            r = read(f0, nf, view(y, (nf, height, width), dt), view(u, (nf, height // 2, width // 2), dt),
                     view(v, (nf, height // 2, width // 2), dt))
            return int(r or 0)
        except BaseException as e:          # noqa: B036 -- handed back to the caller below
            raised.append(e)
            return 1

    def on_write(_user, wp):
        try:
            r = write(StreamWindow(wp.contents, view))
            return int(r or 0)
        except BaseException as e:          # noqa: B036
            raised.append(e)
            return 1

    report = Report() if report is None else report
    rc = call(READ_CB(on_read), WRITE_CB(on_write), ctypes.byref(report))
    if raised:
        try:
            check(rc)
        except PmpError:
            raise raised[0]
    check(rc)
    return report


class StreamWindow:
    """One window of pmp_predict_stream: first_frame, frames, n_qps, report (dict) and, keyed by (qp index, component
    0 luma / 1 chroma), values (int8 [frames * per]) and text (uint8) numpy views of library memory, valid only during
    the write callback.  Results not computed or not asked for are absent."""

    def __init__(self, w, view):
        import numpy as np
        self.first_frame, self.frames, self.n_qps = w.first_frame, w.frames, w.n_qps
        self.report = w.report.as_dict()
        self.values, self.text = {}, {}
        for q in range(w.n_qps):
            for c in range(2):
                if w.values[q][c]:
                    self.values[(q, c)] = view(w.values[q][c], (w.n_values[q][c],), np.int8)
                if w.text[q][c]:
                    self.text[(q, c)] = view(w.text[q][c], (w.text_bytes[q][c],), np.uint8)
