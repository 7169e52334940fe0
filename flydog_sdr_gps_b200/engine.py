"""Python driver over the C ABI (include/acq_b200.h): used by the tests, smoke() and bench.py.

All computation happens in libacq_b200.so on the GPU; this module only marshals numpy / torch buffers.
"""
import ctypes as C

import numpy as np

from . import _lib
from .sats import E1B

N = 16384
BLOCK_BYTES = 8192
BIN_HZ = 249.755859375
LAGS_L1 = 4092
LAGS_E1B = 16368
WRAP_REFERENCE, WRAP_CIRCULAR = 0, 1

RECORD_DTYPE = np.dtype([("sat", "<i4"), ("lag", "<i4"), ("dop", "<i4"),
                         ("peak", "<f4"), ("noise", "<f4"), ("snr", "<f4")])
CELL_DTYPE = np.dtype([("peak", "<f4"), ("noise", "<f4"), ("snr", "<f4"), ("lag", "<i4")])
FINE_DTYPE = np.dtype([("dop_hz", "<f4"), ("code_fs", "<f4"), ("peak", "<f4"), ("ca_shift", "<i4")])
assert RECORD_DTYPE.itemsize == 24 and CELL_DTYPE.itemsize == 16 and FINE_DTYPE.itemsize == 16


class AcqError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("acq error %d: %s" % (code, msg))
        self.code = code


def _check(rc, lib=None):
    if rc != 0:
        raise AcqError(rc, (lib or _lib.load()).acq_last_error().decode())


def default_params(**kw):
    p = _lib.AcqParams()
    _check(_lib.load().acq_params_default(C.byref(p)))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def microbench(device=0):
    """On-device FP32 / shared-memory / L2 micro-benchmarks (roofline denominators)."""
    out = (C.c_double * 8)()
    _check(_lib.load().acq_microbench(device, out, 8))
    keys = ["ffma_tflops", "ffma2_tflops", "smem_tbs", "l2_tbs", "sm_mhz", "fadd_tops", "fadd2_tops"]
    return {k: out[i] for i, k in enumerate(keys)}


class AcqEngine:
    """One engine per GPU.  `sats` is the receiver's satellite table [(prn, t1, t2, type), ...]."""

    def __init__(self, sats, params=None, device=0, variant=None):
        """variant: name of an experiment build of the library (flydog_sdr_gps_b200/_build.py VARIANTS; tests only)."""
        self._L = _lib.load_variant(variant) if variant else _lib.load()
        self.sats = [tuple(int(v) for v in s) for s in sats]
        self.params = params if params is not None else default_params()
        arr = (_lib.AcqSat * len(self.sats))()
        for i, s in enumerate(self.sats):
            arr[i].prn, arr[i].t1, arr[i].t2, arr[i].type = s
        h = C.c_void_p()
        _check(self._L.acq_create(C.byref(h), C.byref(self.params), arr, len(self.sats), device), self._L)
        self._h = h
        self.device = device

    # ---- lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._L.acq_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- properties
    @property
    def n_dop(self):
        return self.params.dop_hi - self.params.dop_lo + 1

    @property
    def k_noncoh(self):
        return self.params.k_noncoh

    @property
    def block_bytes(self):
        """Bytes of one 65536-sample block in this engine's capture format (ACQ_CAPTURE_BLOCK_BYTES)."""
        return 2 * BLOCK_BYTES if self.params.sample_bits == 2 else BLOCK_BYTES

    @property
    def launch_count(self):
        return int(self._L.acq_launch_count(self._h))

    def set_profiling(self, on=True):
        _check(self._L.acq_set_profiling(self._h, 1 if on else 0), self._L)

    def kernel_ms(self):
        """Device time of each kernel of the most recent search (needs set_profiling(True))."""
        out = (C.c_float * 4)()
        _check(self._L.acq_get_kernel_ms(self._h, out, 4), self._L)
        return dict(zip(["front_end", "fwd_fft", "search", "best_dop"], [float(v) for v in out]))

    def device_info(self):
        d, s, c = C.c_int(), C.c_int(), C.c_int()
        _check(self._L.acq_device_info(self._h, C.byref(d), C.byref(s), C.byref(c)), self._L)
        return {"device": d.value, "sm_count": s.value, "sm_clock_khz": c.value}

    def cells_per_search(self, sel=None):
        """Correlation cells (sat x Doppler x lag) examined per capture (SURVEY 8(d) metric)."""
        idx = range(len(self.sats)) if sel is None else sel
        return sum(self.n_dop * (LAGS_E1B if self.sats[i][3] == E1B else LAGS_L1) for i in idx)

    def tiles_per_search(self, sel=None):
        n = len(self.sats) if sel is None else len(sel)
        return n * self.n_dop * self.k_noncoh

    # ---- helpers
    def _sel(self, sel):
        if sel is None:
            return None, len(self.sats), None
        a = np.ascontiguousarray(sel, np.int32)
        return a.ctypes.data_as(C.c_void_p), len(a), a

    def _packed(self, packed):
        a = np.ascontiguousarray(packed, np.uint8).reshape(-1)
        per = self.k_noncoh * self.block_bytes
        if a.size == 0 or a.size % per:
            raise ValueError("packed must hold a whole number of captures of %d bytes" % per)
        return a, a.size // per

    # ---- search over host buffers (the reference-facing call)
    def search(self, packed, sel=None, want_grid=False):
        a, n_cap = self._packed(packed)
        sp, n_sel, keep = self._sel(sel)
        out = np.zeros((n_cap, n_sel), RECORD_DTYPE)
        if want_grid:
            grid = np.zeros((n_cap, n_sel, self.n_dop), CELL_DTYPE)
            _check(self._L.acq_search_grid(self._h, a.ctypes.data, n_cap, sp, n_sel, out.ctypes.data,
                                           grid.ctypes.data), self._L)
            return out, grid
        _check(self._L.acq_search(self._h, a.ctypes.data, n_cap, sp, n_sel, out.ctypes.data), self._L)
        return out

    def search_ptr(self, packed_ptr, n_cap, out_ptr, sel=None):
        """acq_search on raw host pointers (e.g. pinned torch tensors): no allocation on the way."""
        sp, n_sel, keep = self._sel(sel)
        _check(self._L.acq_search(self._h, packed_ptr, n_cap, sp, n_sel, out_ptr), self._L)

    def submit(self, packed, out, sel=None):
        a, n_cap = self._packed(packed)
        sp, n_sel, keep = self._sel(sel)
        assert out.dtype == RECORD_DTYPE and out.size == n_cap * n_sel
        self._keep = (a, keep, out)
        _check(self._L.acq_submit(self._h, a.ctypes.data, n_cap, sp, n_sel, out.ctypes.data), self._L)

    def poll(self):
        rc = self._L.acq_poll(self._h)
        if rc < 0:
            _check(rc, self._L)
        return bool(rc)

    def wait(self):
        _check(self._L.acq_wait(self._h), self._L)

    # ---- device-resident search (torch tensors on this engine's GPU)
    def search_device(self, packed_dev, out_dev, n_cap, sel=None, stream_ptr=None):
        """packed_dev / out_dev: device pointers (ints).  Enqueues on stream_ptr (None = engine stream)."""
        sp, n_sel, keep = self._sel(sel)
        _check(self._L.acq_search_device(self._h, packed_dev, n_cap, sp, n_sel, out_dev, stream_ptr), self._L)

    # ---- aided search: each (capture, satellite) row over its own Doppler window of W = 2 * half_width + 1 indices
    def search_aided(self, packed, dop_center, half_width, sel=None, want_grid=False):
        """acq_search_aided.  dop_center: int [n_cap, n_sel] (or anything of that size), Doppler indices in the engine's
        units; row r searches [lo_r, lo_r + W - 1], lo_r = clamp(center - half_width, dop_lo, dop_hi - 2 half_width).
        Returns records [n_cap, n_sel] (dop absolute) and, if asked, the window cells [n_cap, n_sel, W]."""
        a, n_cap = self._packed(packed)
        sp, n_sel, keep = self._sel(sel)
        c = np.ascontiguousarray(dop_center, np.int32).reshape(-1)
        if c.size != n_cap * n_sel:
            raise ValueError("dop_center must hold n_captures * n_sel = %d centres (got %d)" % (n_cap * n_sel, c.size))
        out = np.zeros((n_cap, n_sel), RECORD_DTYPE)
        grid = np.zeros((n_cap, n_sel, 2 * max(int(half_width), 0) + 1), CELL_DTYPE) if want_grid else None
        _check(self._L.acq_search_aided(self._h, a.ctypes.data, n_cap, sp, n_sel, c.ctypes.data, int(half_width),
                                        out.ctypes.data, grid.ctypes.data if want_grid else None), self._L)
        return (out, grid) if want_grid else out

    def search_aided_device(self, packed_dev, dop_center_dev, half_width, out_dev, n_cap, sel=None, stream_ptr=None):
        """acq_search_aided_device: packed_dev / dop_center_dev (int32, n_cap * n_sel) / out_dev are device pointers
        (ints).  Enqueues on stream_ptr (None = engine stream); the centres are read by the kernels."""
        sp, n_sel, keep = self._sel(sel)
        _check(self._L.acq_search_aided_device(self._h, packed_dev, n_cap, sp, n_sel, dop_center_dev, int(half_width), out_dev,
                                               stream_ptr), self._L)

    def refine(self, records):
        """acq_refine: hand-off refinement of the records of the most recent search()/wait() -- FINE_DTYPE array of
        the same shape (Doppler in Hz from a three-bin interpolation, code phase in FS samples from early/late)."""
        r = np.ascontiguousarray(records, RECORD_DTYPE)
        out = np.zeros(r.shape, FINE_DTYPE)
        _check(self._L.acq_refine(self._h, r.ctypes.data, r.size, out.ctypes.data), self._L)
        return out

    def detected(self, records):
        """Detection rule of SearchTask (search.cpp:549,591) applied to a record array."""
        r = np.asarray(records)
        thr = np.where(np.array([self.sats[s][3] for s in r["sat"].reshape(-1)]).reshape(r.shape) == E1B,
                       self.params.thr_e1b, self.params.thr_l1)
        return r["snr"] >= thr

    # ---- introspection
    def code_spectrum(self, sat):
        out = np.zeros(2 * N, np.float32)
        _check(self._L.acq_get_code_spectrum(self._h, sat, out.ctypes.data), self._L)
        return out.view(np.complex64)

    def capture_spectrum(self, packed_block, half_rot=0):
        a = np.ascontiguousarray(packed_block, np.uint8).reshape(-1)
        assert a.size == self.block_bytes
        x2 = np.zeros(2 * N, np.float32)
        D = np.zeros(2 * N, np.float32)
        _check(self._L.acq_get_capture_spectrum(self._h, a.ctypes.data, half_rot, x2.ctypes.data, D.ctypes.data), self._L)
        return x2.view(np.complex64), D.view(np.complex64)
