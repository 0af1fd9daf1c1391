"""ctypes binding of the C-ABI engine (include/cwt_b200.h).  No PyTorch, no CPU
fallback: if the CUDA library or a device is missing, calls raise EngineError."""
import ctypes
import os
import threading
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcwtb200.so")

MORLET, PAUL, DOG, TABLE = 0, 1, 2, 3
F64, F32 = 0, 1

_P = ctypes.c_void_p
_I64 = ctypes.c_int64
_D = ctypes.c_double
_I = ctypes.c_int


class EngineError(RuntimeError):
    pass


_SIGNATURES = {
    "cwtb_device_count": (_I, []),
    "cwtb_create": (_I, [_I, ctypes.POINTER(_P)]),
    "cwtb_destroy": (None, [_P]),
    "cwtb_last_error": (ctypes.c_char_p, [_P]),
    "cwtb_version": (ctypes.c_char_p, []),
    "cwtb_set_band_eps": (_I, [_P, _D]),
    "cwtb_set_expand_eps": (_I, [_P, _D, _D]),
    "cwtb_set_padding": (_I, [_P, _I]),
    "cwtb_set_smooth_filter": (_I, [_P, _P, _I, _I64]),
    "cwtb_host_alloc": (_I, [_P, ctypes.c_size_t, ctypes.POINTER(_P)]),
    "cwtb_host_free": (_I, [_P, _P]),
    "cwtb_cwt": (_I, [_P, _P, _I, _I64, _D, _P, _I, _I, _D, _I, _P]),
    "cwtb_cwt_dev": (_I, [_P, _P, _I, _I64, _D, _P, _I, _I, _D, _I]),
    "cwtb_get_w": (_I, [_P, _P, _I, _I, _I]),
    "cwtb_get_signal_fft": (_I, [_P, _P]),
    "cwtb_padded_length": (_I64, [_P]),
    "cwtb_job_serial": (_I64, [_P]),
    "cwtb_w_device_ptr": (_P, [_P]),
    "cwtb_last_kernel_ms": (_D, [_P]),
    "cwtb_last_launch_count": (_I, [_P]),
    "cwtb_last_plan": (_I, [_P, _P, _I]),
    "cwtb_bench_last": (_I, [_P, _I, ctypes.POINTER(_D)]),
    "cwtb_profile_last": (_I, [_P, ctypes.c_char_p, ctypes.c_size_t]),
    "cwtb_profile_begin": (_I, [_P]),
    "cwtb_profile_end": (_I, [_P, ctypes.c_char_p, ctypes.c_size_t]),
    "cwtb_dev_alloc": (_I, [_P, ctypes.c_size_t, ctypes.POINTER(_P)]),
    "cwtb_dev_free": (_I, [_P, _P]),
    "cwtb_memcpy_h2d": (_I, [_P, _P, _P, ctypes.c_size_t]),
    "cwtb_memcpy_d2h": (_I, [_P, _P, _P, ctypes.c_size_t]),
    "cwtb_sync": (_I, [_P]),
    "cwtb_fft_c2c": (_I, [_P, _P, _P, _I64, _I, _I, _I]),
    "cwtb_cwt_to_host": (_I, [_P, _P, _I, _I64, _D, _P, _I, _I, _D, _I, _P, _I]),
    "cwtb_icwt_sum": (_I, [_P, _P]),
    "cwtb_icwt_sum_host": (_I, [_P, _P, _P, _I, _I64, _P]),
    "cwtb_get_power": (_I, [_P, _P]),
    "cwtb_global_power": (_I, [_P, _P]),
    "cwtb_get_power_scaled": (_I, [_P, _P, _P]),
    "cwtb_global_power_ranges": (_I, [_P, _P, _P, _P]),
    "cwtb_scale_avg_power": (_I, [_P, _P, _P]),
    "cwtb_xwt": (_I, [_P, _P, _P, _I64, _D, _P, _I, _I, _D, _P]),
    "cwtb_wct": (_I, [_P, _P, _P, _I64, _D, _D, _P, _I, _I, _D, _I, _P, _P]),
    "cwtb_smooth": (_I, [_P, _P, _I, _I, _I64, _D, _P, _I, _P]),
    "cwtb_wct_mc": (_I, [_P, _P, _I, _I64, _D, _D, _P, _I, _I, _D, _I, _P, _I, _I, _P]),
    "cwtb_wct_mc_seeded": (_I, [_P, ctypes.c_uint64, _I64, _I, _I64, _D, _P, _I, _I, _D, _I, _P, _I, _I, _P]),
    "cwtb_mc_surrogates": (_I, [_P, ctypes.c_uint64, _I64, _I, _I64, _P]),
    "cwtb_cwt_batch": (_I, [_P, _P, _I, _I, _I64, _D, _P, _I, _I, _D, _I, _P, _P]),
    "cwtb_cwt_batch_dev": (_I, [_P, _P, _I, _I64, _D, _P, _I, _I, _D, _I, _P]),
    "cwtb_cwt_batch_products": (_I, [_P, _P, _I, _I, _I64, _D, _P, _I, _I, _D, _I, _P, _P, _I, _P, _P,
                                     _D, _D, _I, _P, _P, _P, _P]),
    "cwtb_comm_unique_id": (_I, [_P]),
    "cwtb_comm_init": (_I, [_P, _I, _I, _P]),
    "cwtb_comm_destroy": (_I, [_P]),
    "cwtb_comm_world": (_I, [_P]),
    "cwtb_comm_rank": (_I, [_P]),
    "cwtb_comm_allgather": (_I, [_P, _P, _P, ctypes.c_size_t]),
    "cwtb_comm_allreduce_sum_i64": (_I, [_P, _P, ctypes.c_size_t]),
    "cwtb_comm_allreduce_max_f64": (_I, [_P, _P, ctypes.c_size_t]),
    "cwtb_comm_broadcast": (_I, [_P, _P, ctypes.c_size_t, _I]),
}


def load_library(path=None):
    """dlopen the engine and declare the prototypes of every exported symbol."""
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise EngineError(
            "CUDA engine not built: %s is missing (run `python -m pycwt_b200.build`)" % path)
    lib = ctypes.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


def _ptr(a):
    return a.ctypes.data_as(_P)


def _locked(method):
    """Run an Engine method under the engine's (re-entrant) lock."""
    import functools

    @functools.wraps(method)
    def wrapper(self, *args, **kwargs):
        with self.lock:
            return method(self, *args, **kwargs)
    return wrapper


class Engine(object):
    """One context = one device + one stream.  Every call into the C library is made under
    `self.lock`, a re-entrant lock: compound operations of the Python surface (set the length
    policy, transform, fetch the coefficients, fetch the spectrum) hold it across all their
    steps, so concurrent callers of the shared default engine cannot interleave inside one
    another's transform (the C side keeps ONE resident job per context)."""

    def __init__(self, device=0, lib_path=None):
        self.lib = load_library(lib_path)
        if self.lib.cwtb_device_count() <= 0:
            raise EngineError("no CUDA device visible: the B200 engine has no CPU fallback")
        h = _P()
        rc = self.lib.cwtb_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise EngineError("cwtb_create(device=%d) failed with status %d" % (device, rc))
        self.h = h
        self.device = device
        self.lock = threading.RLock()
        # pinned result buffers: bookkeeping has its own small lock because buffers come back
        # from weakref finalizers on arbitrary threads (re-entrant: a finalizer may run at any
        # allocation point of the thread that already holds it)
        self._pool_lock = threading.RLock()
        self._pool = []          # idle pinned buffers, least recently released first: (nbytes, addr)
        self._pool_bytes = 0
        self._dead = []          # retired pinned buffers waiting for _reap()
        self._outstanding = 0    # result arrays still alive that alias pinned memory

    def _reap(self):
        """Free the pinned buffers the finalizers retired.  Finalizers never call into the
        library themselves (they can fire at any allocation point of any thread, also inside
        this class's critical sections); the frees happen here, under the engine lock."""
        with self._pool_lock:
            dead, self._dead = self._dead, []
        if dead and getattr(self, "h", None):
            with self.lock:
                for addr in dead:
                    self.lib.cwtb_host_free(self.h, _P(addr))

    def trim(self, keep_bytes=0):
        """Release idle pinned result buffers until at most `keep_bytes` stay pooled."""
        with self._pool_lock:
            while self._pool and self._pool_bytes > keep_bytes:
                nbytes, addr = self._pool.pop(0)
                self._pool_bytes -= nbytes
                self._dead.append(addr)
        self._reap()

    def close(self):
        """Destroy the context.  While result arrays that alias its pinned memory are alive
        only the idle pooled buffers are released; the context goes with the last array."""
        if not getattr(self, "h", None):
            return
        with self.lock:
            self._closing = True
            self.trim(0)
            if self._outstanding == 0:
                self.lib.cwtb_destroy(self.h)
                self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.cwtb_last_error(self.h)
            raise EngineError("engine status %d: %s" % (rc, (msg or b"").decode()))

    def version(self):
        return self.lib.cwtb_version().decode()

    # (rows, n0) of the transform the device holds, when the last call left a single well-defined
    # one there; the fetch/reduction methods check their arguments against it because the C side
    # sizes its copies from the resident job, not from the caller's arrays
    _resident = None

    def _expect_resident(self, rows=None, n0=None):
        if self._resident is None:
            return
        r, n = self._resident
        if (rows is not None and rows != r) or (n0 is not None and n0 != n):
            raise ValueError("the resident transform is %d x %d, the call asks for %s x %s"
                             % (r, n, "?" if rows is None else rows, "?" if n0 is None else n0))

    @_locked
    def set_band_eps(self, eps):
        self._check(self.lib.cwtb_set_band_eps(self.h, float(eps)))

    @_locked
    def set_expand_eps(self, eps64=5e-13, eps32=2e-7):
        """Tolerance of the band-limited expansion path (include/cwt_b200.h); 0 switches it off
        (every scale through the exact pruned transforms)."""
        self._check(self.lib.cwtb_set_expand_eps(self.h, float(eps64), float(eps32)))

    @_locked
    def set_smooth_filter(self, table=None):
        """Real frequency responses [rows, n] of the time smoothing used by smooth / wct / wct_mc
        instead of Morlet's Gaussian; None restores the Gaussian."""
        if table is None:
            self._check(self.lib.cwtb_set_smooth_filter(self.h, None, 0, 0))
            return
        t = np.ascontiguousarray(table, dtype=np.float64)
        self._check(self.lib.cwtb_set_smooth_filter(self.h, _ptr(t), t.shape[0], t.shape[1]))

    @_locked
    def set_padding(self, pad_to_pow2):
        """True (default): pad to the next power of two like the reference's scipy branch;
        False: transform at the signal's own length (the reference's pyfftw policy)."""
        self._check(self.lib.cwtb_set_padding(self.h, 1 if pad_to_pow2 else 0))
        self._pad_pow2 = bool(pad_to_pow2)

    # ---- pinned host arrays -------------------------------------------------------
    @_locked
    def pinned_empty(self, shape, dtype):
        """numpy array backed by page-locked memory owned by the engine context."""
        dtype = np.dtype(dtype)
        n = int(np.prod(shape)) * dtype.itemsize
        p = _P()
        self._check(self.lib.cwtb_host_alloc(self.h, max(n, 1), ctypes.byref(p)))
        buf = (ctypes.c_char * max(n, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
        return arr, p

    @_locked
    def pinned_free(self, p):
        self.lib.cwtb_host_free(self.h, p)

    #: results at least this large are returned in page-locked memory (D2H at PCIe speed)
    PINNED_MIN_BYTES = 1 << 20
    #: idle pinned memory kept for reuse (env CWTB_POOL_MB).  Default: room for one result of
    #: the north-star size (4.3 GB) so that steady-state calls neither allocate nor pin; least
    #: recently released buffers of any size are evicted first.
    POOL_MAX_BYTES = int(os.environ.get("CWTB_POOL_MB", "4608")) << 20
    _closing = False

    def result_array(self, shape, dtype):
        """Array for a transform result.  Large results alias pinned host memory taken
        from a per-engine pool; the buffer returns to the pool when the array (and every
        view of it) is garbage-collected, so steady-state calls neither allocate nor pin."""
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        nbytes = count * dtype.itemsize
        if nbytes < self.PINNED_MIN_BYTES:
            return np.empty(shape, dtype=dtype)
        self._reap()
        addr = None
        with self._pool_lock:
            for i in range(len(self._pool) - 1, -1, -1):     # most recently released first
                if self._pool[i][0] == nbytes:
                    addr = self._pool.pop(i)[1]
                    self._pool_bytes -= nbytes
                    break
        if addr is None:
            p = _P()
            with self.lock:
                rc = self.lib.cwtb_host_alloc(self.h, nbytes, ctypes.byref(p))
            if rc != 0 or not p.value:
                self.trim(0)      # give pooled buffers of other sizes back and retry once
                with self.lock:
                    rc = self.lib.cwtb_host_alloc(self.h, nbytes, ctypes.byref(p))
            if rc != 0 or not p.value:
                # page-locked memory exhausted: an ordinary array still works, the copy is slower
                return np.empty(shape, dtype=dtype)
            addr = p.value
        buf = (ctypes.c_char * nbytes).from_address(addr)
        with self._pool_lock:
            self._outstanding += 1
        fin = weakref.finalize(buf, self._release, nbytes, addr)
        fin.atexit = False
        return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)

    def _release(self, nbytes, addr):
        """Finalizer of a pinned result array (any thread, any time): pool the buffer and
        retire the least recently released ones beyond POOL_MAX_BYTES.  No library calls."""
        with self._pool_lock:
            self._outstanding -= 1
            last = self._outstanding == 0
            if self.h is None:
                return
            if self._closing or nbytes > self.POOL_MAX_BYTES:
                self._dead.append(addr)
            else:
                self._pool.append((nbytes, addr))
                self._pool_bytes += nbytes
                while self._pool_bytes > self.POOL_MAX_BYTES and len(self._pool) > 1:
                    nb, ad = self._pool.pop(0)
                    self._pool_bytes -= nb
                    self._dead.append(ad)
        if self._closing and last and self.lock.acquire(blocking=False):
            try:
                self.close()
            finally:
                self.lock.release()

    # ---- transform ------------------------------------------------------------------
    @_locked
    def cwt(self, signal, dt, scales, family, param, precision=F64, table=None,
            fetch=True, out_f64=True):
        sig = np.ascontiguousarray(signal)
        if sig.dtype == np.float32:
            is32 = 1
        else:
            sig = np.ascontiguousarray(sig, dtype=np.float64)
            is32 = 0
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        tptr = None
        if table is not None:
            table = np.ascontiguousarray(table, dtype=np.complex128)
            tptr = _ptr(table)
        with self.lock:
            if fetch and table is None:
                # transform and copy back in one call: the engine starts the device->host copy
                # of the rows that are finished first while the remaining kernels still run
                dtype = np.complex128 if (precision == F64 or out_f64) else np.complex64
                W = self.result_array((sj.size, sig.size), dtype)
                self._check(self.lib.cwtb_cwt_to_host(self.h, _ptr(sig), is32, sig.size, float(dt),
                                                      _ptr(sj), sj.size, int(family), float(param),
                                                      int(precision), _ptr(W), 1 if out_f64 else 0))
                self._resident_n0 = sig.size
                self._resident = (sj.size, sig.size)
                return W
            self._check(self.lib.cwtb_cwt(self.h, _ptr(sig), is32, sig.size, float(dt),
                                          _ptr(sj), sj.size, int(family), float(param),
                                          int(precision), tptr))
            self._resident_n0 = sig.size
            self._resident = (sj.size, sig.size)
            if not fetch:
                return None
            return self.get_w(sj.size, sig.size, precision, out_f64)

    @_locked
    def get_w(self, nrows, n0, precision=F64, out_f64=True):
        dtype = np.complex128 if (precision == F64 or out_f64) else np.complex64
        self._expect_resident(None, n0)
        if self._resident is not None and nrows > self._resident[0]:
            raise ValueError("get_w: %d rows requested, %d resident" % (nrows, self._resident[0]))
        W = self.result_array((nrows, n0), dtype)
        self._check(self.lib.cwtb_get_w(self.h, _ptr(W), 1 if out_f64 else 0, 0, nrows))
        return W

    @_locked
    def signal_fft(self):
        npad = int(self.lib.cwtb_padded_length(self.h))
        out = np.empty(max(npad // 2 - 1, 0), dtype=np.complex128)
        if out.size:
            self._check(self.lib.cwtb_get_signal_fft(self.h, _ptr(out)))
        return out

    @_locked
    def job_serial(self):
        return int(self.lib.cwtb_job_serial(self.h))

    @_locked
    def padded_length(self):
        return int(self.lib.cwtb_padded_length(self.h))

    @_locked
    def last_plan(self, n):
        out = (ctypes.c_int * n)()
        m = self.lib.cwtb_last_plan(self.h, out, n)
        return list(out)[:max(m, 0)]

    @_locked
    def last_kernel_ms(self):
        return float(self.lib.cwtb_last_kernel_ms(self.h))

    @_locked
    def last_launch_count(self):
        return int(self.lib.cwtb_last_launch_count(self.h))

    @_locked
    def fft_c2c(self, x, sign, precision=F64):
        x = np.ascontiguousarray(x, dtype=np.complex128)
        if x.ndim == 1:
            x = x[None, :]
        out = np.empty_like(x)
        self._check(self.lib.cwtb_fft_c2c(self.h, _ptr(x), _ptr(out), x.shape[1],
                                          x.shape[0], int(sign), int(precision)))
        return out

    # ---- reductions / derived products of the resident transform ------------------------
    @_locked
    def icwt_sum(self, W=None, scales=None):
        """sum_j Re(W[j, :]) / sqrt(s_j): of the resident transform (W is None) or of a host
        array W[S, n]."""
        with self.lock:
            if W is None:
                n0 = self._resident_n0
                out = self.result_array((n0,), np.float64)     # pinned when large: D2H at PCIe speed
                self._check(self.lib.cwtb_icwt_sum(self.h, _ptr(out)))
                return out
            W = np.ascontiguousarray(W, dtype=np.complex128)
            sj = np.ascontiguousarray(scales, dtype=np.float64)
            out = np.empty(W.shape[1], dtype=np.float64)
            self._check(self.lib.cwtb_icwt_sum_host(self.h, _ptr(W), _ptr(sj), W.shape[0],
                                                    W.shape[1], _ptr(out)))
            return out

    @_locked
    def global_power(self, nrows):
        self._expect_resident(nrows)
        out = np.empty(nrows, dtype=np.float64)
        self._check(self.lib.cwtb_global_power(self.h, _ptr(out)))
        return out

    @_locked
    def global_power_ranges(self, lo, hi):
        """Row means of |W|^2 over the column ranges [lo[j], hi[j]) (NaN where empty)."""
        lo = np.ascontiguousarray(lo, dtype=np.int64)
        hi = np.ascontiguousarray(hi, dtype=np.int64)
        if lo.shape != hi.shape:
            raise ValueError("global_power_ranges: lo and hi must have one entry per row")
        self._expect_resident(lo.size)
        out = np.empty(lo.size, dtype=np.float64)
        with self.lock:
            self._check(self.lib.cwtb_global_power_ranges(self.h, _ptr(lo), _ptr(hi), _ptr(out)))
        return out

    @_locked
    def power(self, nrows, n0, row_scale=None):
        """|W|^2 of the resident transform, optionally times one factor per row."""
        self._expect_resident(nrows, n0)
        out = self.result_array((nrows, n0), np.float64)
        with self.lock:
            if row_scale is None:
                self._check(self.lib.cwtb_get_power(self.h, _ptr(out)))
            else:
                rs = np.ascontiguousarray(row_scale, dtype=np.float64)
                if rs.size != nrows:
                    raise ValueError("power: one factor per row expected")
                self._check(self.lib.cwtb_get_power_scaled(self.h, _ptr(rs), _ptr(out)))
        return out

    @_locked
    def scale_avg_power(self, weights):
        """sum_j weights[j] |W[j, :]|^2 of the resident transform (TC98 eq. 24)."""
        w = np.ascontiguousarray(weights, dtype=np.float64)
        self._expect_resident(w.size)
        out = self.result_array((self._resident_n0,), np.float64)
        with self.lock:
            self._check(self.lib.cwtb_scale_avg_power(self.h, _ptr(w), _ptr(out)))
        return out

    # ---- cross wavelet / coherence ------------------------------------------------------
    @_locked
    def xwt(self, y1, y2, dt, scales, family, param):
        y1 = np.ascontiguousarray(y1, dtype=np.float64)
        y2 = np.ascontiguousarray(y2, dtype=np.float64)
        if y1.shape != y2.shape or y1.ndim != 1:
            raise ValueError("xwt: the two series must be 1-D and of equal length")
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        out = self.result_array((sj.size, y1.size), np.complex128)
        with self.lock:
            self._check(self.lib.cwtb_xwt(self.h, _ptr(y1), _ptr(y2), y1.size, float(dt), _ptr(sj),
                                          sj.size, int(family), float(param), _ptr(out)))
            self._resident_n0 = y1.size
            self._resident = (sj.size, y1.size)     # W12 stays on the device
        return out

    @_locked
    def wct(self, y1, y2, dt, dj, scales, family, param, boxcar_len, want_angle=True):
        y1 = np.ascontiguousarray(y1, dtype=np.float64)
        y2 = np.ascontiguousarray(y2, dtype=np.float64)
        if y1.shape != y2.shape or y1.ndim != 1:
            raise ValueError("wct: the two series must be 1-D and of equal length")
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        WCT = self.result_array((sj.size, y1.size), np.float64)
        aWCT = self.result_array((sj.size, y1.size), np.float64) if want_angle else None
        with self.lock:
            self._check(self.lib.cwtb_wct(self.h, _ptr(y1), _ptr(y2), y1.size, float(dt), float(dj),
                                          _ptr(sj), sj.size, int(family), float(param),
                                          int(boxcar_len), _ptr(WCT),
                                          _ptr(aWCT) if want_angle else None))
            self._resident = None                   # several intermediates, no single transform
        return WCT, aWCT

    @_locked
    def smooth(self, W, dt, scales, boxcar_len):
        W = np.ascontiguousarray(W)
        is_c = np.iscomplexobj(W)
        W = np.ascontiguousarray(W, dtype=np.complex128 if is_c else np.float64)
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        if W.ndim != 2 or sj.ndim != 1 or sj.size != W.shape[0]:
            # the reference fails here too (broadcast of the [S, 1] filter against W, mothers.py:87)
            raise ValueError("smooth: W must be [scales, time] with one scale per row "
                             "(got W %s, %d scales)" % (W.shape, sj.size))
        out = np.empty_like(W)
        with self.lock:
            self._check(self.lib.cwtb_smooth(self.h, _ptr(W), int(is_c), W.shape[0], W.shape[1],
                                             float(dt), _ptr(sj), int(boxcar_len), _ptr(out)))
        return out

    @_locked
    def wct_mc(self, noise, dt, dj, scales, family, param, boxcar_len, mask, maxscale, nbins,
               hist):
        noise = np.ascontiguousarray(noise, dtype=np.float64)
        assert noise.ndim == 3 and noise.shape[1] == 2
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        assert mask.shape == (sj.size, noise.shape[2])
        assert hist.dtype == np.int64 and hist.flags.c_contiguous and hist.shape == (sj.size, nbins)
        with self.lock:
            self._check(self.lib.cwtb_wct_mc(self.h, _ptr(noise), noise.shape[0], noise.shape[2],
                                             float(dt), float(dj), _ptr(sj), sj.size, int(family),
                                             float(param), int(boxcar_len), _ptr(mask),
                                             int(maxscale), int(nbins), _ptr(hist)))
            self._resident = None
        return hist

    @_locked
    def wct_mc_seeded(self, seed, first_pair, n_pairs, n0, dt, scales, family, param, boxcar_len, mask,
                      maxscale, nbins, hist):
        """Monte-Carlo coherence histograms of `n_pairs` surrogate pairs drawn on the device
        (Philox stream keyed by (seed, pair number)); accumulated into `hist`."""
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        mask = np.ascontiguousarray(mask, dtype=np.uint8)
        assert mask.shape == (sj.size, int(n0))
        assert hist.dtype == np.int64 and hist.flags.c_contiguous and hist.shape == (sj.size, nbins)
        self._check(self.lib.cwtb_wct_mc_seeded(self.h, int(seed) & (2 ** 64 - 1), int(first_pair), int(n_pairs),
                                                int(n0), float(dt), _ptr(sj), sj.size, int(family),
                                                float(param), int(boxcar_len), _ptr(mask), int(maxscale),
                                                int(nbins), _ptr(hist)))
        self._resident = None
        return hist

    @_locked
    def mc_surrogates(self, seed, first_pair, n_pairs, n0):
        out = np.empty((int(n_pairs), 2, int(n0)), dtype=np.float64)
        self._check(self.lib.cwtb_mc_surrogates(self.h, int(seed) & (2 ** 64 - 1), int(first_pair),
                                                int(n_pairs), int(n0), _ptr(out)))
        return out

    @_locked
    def cwt_batch(self, X, dt, scales, family, param, precision=F64, want_power=True,
                  want_w=False):
        X = np.ascontiguousarray(X)
        if X.dtype != np.float32:
            X = np.ascontiguousarray(X, dtype=np.float64)
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        nch, n0 = X.shape
        power = np.empty((nch, sj.size), dtype=np.float64) if want_power else None
        W = None
        if want_w:
            W = np.empty((nch, sj.size, n0), dtype=np.complex128 if precision == F64 else np.complex64)
        with self.lock:
            self._check(self.lib.cwtb_cwt_batch(self.h, _ptr(X), int(X.dtype == np.float32), nch, n0,
                                                float(dt), _ptr(sj), sj.size, int(family),
                                                float(param), int(precision),
                                                _ptr(power) if want_power else None,
                                                _ptr(W) if want_w else None))
            self._resident = None                   # the last chunk of channels only
        return power, W

    @_locked
    def cwt_batch_products(self, X, dt, scales, family, param, precision=F64, coi_ranges=None,
                           band_weights=None, chan_scale=None, icwt_factor=None):
        """Batched transform of the rows of X [C, n0] with per-channel products reduced on the
        device (cwtb_cwt_batch_products).  coi_ranges: (lo, hi) int64 per scale; band_weights:
        [n_bands, S]; chan_scale: C factors of the band powers; icwt_factor: real or complex
        (the type of the icwt output).  Returns (power [C, S], power_coi [C, S] or None,
        band [C, n_bands, n0] or None, icwt [C, n0] or None)."""
        X = np.ascontiguousarray(X)
        if X.dtype != np.float32:
            X = np.ascontiguousarray(X, dtype=np.float64)
        if X.ndim != 2:
            raise ValueError("cwt_batch_products: X must be [channels, samples]")
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        nch, n0 = X.shape
        power = np.empty((nch, sj.size), dtype=np.float64)
        lo = hi = power_coi = None
        if coi_ranges is not None:
            lo = np.ascontiguousarray(coi_ranges[0], dtype=np.int64)
            hi = np.ascontiguousarray(coi_ranges[1], dtype=np.int64)
            if lo.shape != (sj.size,) or hi.shape != (sj.size,):
                raise ValueError("cwt_batch_products: one COI range per scale expected")
            power_coi = np.empty((nch, sj.size), dtype=np.float64)
        wt = band = None
        nb = 0
        if band_weights is not None:
            wt = np.ascontiguousarray(band_weights, dtype=np.float64)
            if wt.ndim != 2 or wt.shape[1] != sj.size:
                raise ValueError("cwt_batch_products: band weights must be [n_bands, scales]")
            nb = wt.shape[0]
            if nb > 0:
                band = self.result_array((nch, nb, n0), np.float64)   # pinned when large: async copies
        cs = None
        if chan_scale is not None:
            cs = np.ascontiguousarray(chan_scale, dtype=np.float64)
            if cs.shape != (nch,):
                raise ValueError("cwt_batch_products: one channel factor per channel expected")
        want, fac, iw = 0, 0j, None
        if icwt_factor is not None:
            fac = complex(icwt_factor)
            want = 2 if np.iscomplexobj(icwt_factor) else 1
            iw = self.result_array((nch, n0), np.complex128 if want == 2 else np.float64)
        with self.lock:
            self._check(self.lib.cwtb_cwt_batch_products(
                self.h, _ptr(X), int(X.dtype == np.float32), nch, n0, float(dt), _ptr(sj), sj.size,
                int(family), float(param), int(precision),
                _ptr(lo) if lo is not None else None, _ptr(hi) if hi is not None else None,
                nb, _ptr(wt) if nb else None, _ptr(cs) if cs is not None else None,
                fac.real, fac.imag, want, _ptr(power),
                _ptr(power_coi) if power_coi is not None else None,
                _ptr(band) if band is not None else None, _ptr(iw) if iw is not None else None))
            self._resident = None                   # the last chunk of channels only
        return power, power_coi, band, iw

    # ---- device-resident benchmarking helpers -------------------------------------
    @_locked
    def dev_alloc(self, nbytes):
        p = _P()
        self._check(self.lib.cwtb_dev_alloc(self.h, nbytes, ctypes.byref(p)))
        return p

    @_locked
    def dev_free(self, p):
        self.lib.cwtb_dev_free(self.h, p)

    @_locked
    def h2d(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self._check(self.lib.cwtb_memcpy_h2d(self.h, dptr, _ptr(arr), arr.nbytes))

    @_locked
    def cwt_dev(self, dptr, is_f32, n0, dt, scales, family, param, precision=F64):
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        self._check(self.lib.cwtb_cwt_dev(self.h, dptr, int(is_f32), int(n0), float(dt),
                                          _ptr(sj), sj.size, int(family), float(param),
                                          int(precision)))
        self._resident_n0 = int(n0)
        self._resident = (sj.size, int(n0))

    @_locked
    def cwt_batch_dev(self, dptr, n_chan, n0, dt, scales, family, param, precision=F64,
                      want_power=False):
        sj = np.ascontiguousarray(scales, dtype=np.float64)
        power = np.empty((n_chan, sj.size), dtype=np.float64) if want_power else None
        self._check(self.lib.cwtb_cwt_batch_dev(self.h, dptr, int(n_chan), int(n0), float(dt),
                                                _ptr(sj), sj.size, int(family), float(param),
                                                int(precision), _ptr(power) if want_power else None))
        self._resident_n0 = int(n0)
        self._resident = (int(n_chan) * sj.size, int(n0))
        return power

    @_locked
    def bench_last(self, iters):
        ms = _D()
        self._check(self.lib.cwtb_bench_last(self.h, int(iters), ctypes.byref(ms)))
        return ms.value

    @_locked
    def profile_last(self):
        """Per-kernel-type device times of one pass of the last cwt_dev transform:
        list of dicts {name, launches, ms, rows}."""
        buf = ctypes.create_string_buffer(1 << 16)
        n = self.lib.cwtb_profile_last(self.h, buf, len(buf))
        if n < 0:
            self._check(n)
        out = []
        for line in buf.value.decode().splitlines():
            name, nl, ms, rows = line.rsplit("|", 3)
            out.append({"name": name, "launches": int(nl), "ms": float(ms), "rows": int(rows)})
        return out

    @staticmethod
    def _parse_profile(text):
        out = []
        for line in text.splitlines():
            name, nl, ms, rows = line.rsplit("|", 3)
            out.append({"name": name, "launches": int(nl), "ms": float(ms), "rows": int(rows)})
        return out

    @_locked
    def profile_begin(self):
        """Start recording per-kernel device times of every following call (serialised streams)."""
        self._check(self.lib.cwtb_profile_begin(self.h))

    @_locked
    def profile_end(self):
        buf = ctypes.create_string_buffer(1 << 16)
        n = self.lib.cwtb_profile_end(self.h, buf, len(buf))
        if n < 0:
            self._check(n)
        return self._parse_profile(buf.value.decode())

    @_locked
    def sync(self):
        self._check(self.lib.cwtb_sync(self.h))

    # ---- multi-GPU collectives (NCCL behind the C ABI; no torch) --------------------
    def comm_unique_id(self):
        """128-byte NCCL id (rank 0 creates it, the host program distributes it)."""
        buf = ctypes.create_string_buffer(128)
        rc = self.lib.cwtb_comm_unique_id(buf)
        if rc != 0:
            raise EngineError("cwtb_comm_unique_id failed with status %d (libnccl not loadable?)" % rc)
        return buf.raw

    @_locked
    def comm_init(self, world, rank, uid):
        buf = ctypes.create_string_buffer(bytes(uid), 128)
        self._check(self.lib.cwtb_comm_init(self.h, int(world), int(rank), buf))

    @_locked
    def comm_destroy(self):
        self.lib.cwtb_comm_destroy(self.h)

    def comm_world(self):
        return int(self.lib.cwtb_comm_world(self.h))

    def comm_rank(self):
        return int(self.lib.cwtb_comm_rank(self.h))

    @_locked
    def comm_allgather(self, local):
        """Every rank contributes an equal-shape array; returns the [world, ...] stack."""
        local = np.ascontiguousarray(local)
        out = np.empty((self.comm_world(),) + local.shape, dtype=local.dtype)
        self._check(self.lib.cwtb_comm_allgather(self.h, _ptr(local), _ptr(out), local.nbytes))
        return out

    @_locked
    def comm_allreduce_sum(self, array):
        a = np.ascontiguousarray(array, dtype=np.int64).copy()
        self._check(self.lib.cwtb_comm_allreduce_sum_i64(self.h, _ptr(a), a.size))
        return a

    @_locked
    def comm_allreduce_max(self, array):
        a = np.atleast_1d(np.ascontiguousarray(array, dtype=np.float64)).copy()
        self._check(self.lib.cwtb_comm_allreduce_max_f64(self.h, _ptr(a), a.size))
        return a

    @_locked
    def comm_broadcast(self, array, root=0):
        a = np.ascontiguousarray(array).copy()
        self._check(self.lib.cwtb_comm_broadcast(self.h, _ptr(a), a.nbytes, int(root)))
        return a


_default = {}
_default_lock = threading.Lock()


def device_count():
    return int(load_library().cwtb_device_count())


def default_engine(device=None):
    """Process-wide engine per device (device from CWTB_DEVICE / LOCAL_RANK, default 0)."""
    if device is None:
        device = int(os.environ.get("CWTB_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _default_lock:
        if device not in _default:
            _default[device] = Engine(device)
        return _default[device]
