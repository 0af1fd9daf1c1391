"""Device-resident transform and its derived products (SURVEY 8f rank 2).

`pycwt.cwt` has to hand the caller a complex128 array of S x N coefficients; at the north-star
size that is 4.3 GB over PCIe for 2.3 ms of GPU work.  What the reference's sample scripts
then do with W (pycwt/sample/simple_sample.py:64-96) are reductions of |W|^2:

    power        = |W|^2                      (optionally rectified: / s_j, Liu et al. 2007,
                                               docs/tutorial/cwt.md:49-53)
    glbl_power   = power.mean(axis=1)         (simple_sample.py:79)
    scale_avg    = dj*dt/Cdelta * sum_{j in band} power[j] / s_j      (:88-91, TC98 eq. 24)
    iwave        = icwt(W, ...)               (:60)

`cwt_resident` runs the same transform as `cwt` but keeps W in HBM and returns a handle whose
methods evaluate those products on the device, so only O(S) or O(N) numbers cross the bus.
The handle is valid until the next transform on the same engine.
"""
import numpy as np

from . import _engine
from .helpers import fft, fft_kwargs
from .wavelet import (_check_parameter_wavelet, _nan_rows, _precision, _resolve_scales,
                      _sync_padding)

__all__ = ['cwt_resident', 'ResidentTransform']


def _live(method):
    """Product methods run as one engine transaction: check that this transform is still the
    resident one and evaluate, under the engine lock."""
    import functools

    @functools.wraps(method)
    def wrapper(self, *args, **kwargs):
        with self.engine.lock:
            self._check_live()
            return method(self, *args, **kwargs)
    return wrapper


def coi_ranges(wavelet, n0, dt, period):
    """Columns inside the cone of influence of an n0-sample series, per period: period_j <= coi[n]
    holds on one centred range [lo_j, hi_j) (empty ranges have lo_j == hi_j)."""
    c = wavelet.flambda() * wavelet.coi() * dt
    # coi[n] = c * (n0/2 - |n - (n0-1)/2|) >= period  <=>  |n - (n0-1)/2| <= n0/2 - period/c
    half = n0 / 2 - np.asarray(period) / c
    mid = (n0 - 1) / 2
    lo = np.ceil(mid - half - 1e-12).astype(np.int64)
    hi = np.floor(mid + half + 1e-12).astype(np.int64) + 1
    empty = half < 0
    lo = np.clip(lo, 0, n0)
    hi = np.clip(hi, 0, n0)
    hi[empty] = lo[empty]
    return lo, hi


def coi_curve(wavelet, n0, dt):
    """The cone of influence of an n0-sample series, as `cwt` returns it (wavelet.py:118-120)."""
    coi = (n0 / 2 - np.abs(np.arange(0, n0) - (n0 - 1) / 2))
    return wavelet.flambda() * wavelet.coi() * dt * coi


class ResidentTransform(object):
    """W[S, n0] of one `cwt_resident` call, resident on the device."""

    def __init__(self, engine, wavelet, n0, dt, dj, sj, freqs, precision, serial):
        self.engine = engine
        self.wavelet = wavelet
        self.n0 = int(n0)
        self.dt = float(dt)
        self.dj = dj
        self.scales = sj
        self.freqs = freqs
        self.precision = precision
        self._serial = serial
        self.npad = fft_kwargs(range(self.n0))['n']       # transform length (helpers.py:15-30)
        self._coi = None
        self._fftfreqs = None

    # O(n0) host arrays of the `cwt` return tuple, built on first use
    @property
    def coi(self):
        if self._coi is None:
            self._coi = coi_curve(self.wavelet, self.n0, self.dt)
        return self._coi

    @property
    def fftfreqs(self):
        if self._fftfreqs is None:
            npad = self.npad
            self._fftfreqs = (2 * np.pi * fft.fftfreq(npad, self.dt))[1:npad // 2] / (2 * np.pi)
        return self._fftfreqs

    # -- bookkeeping ---------------------------------------------------------------------
    def _check_live(self):
        if self.engine.job_serial() != self._serial:
            raise _engine.EngineError("this transform is no longer resident: another transform "
                                      "has run on the same engine")

    @property
    def shape(self):
        return (len(self.scales), self.n0)

    @property
    def period(self):
        return 1.0 / np.asarray(self.freqs)

    # -- the products --------------------------------------------------------------------
    @_live
    def wave(self):
        """The coefficients themselves (complex128, S x n0): the expensive fetch."""
        return self.engine.get_w(len(self.scales), self.n0, self.precision)

    @_live
    def fft(self):
        """Normalised signal spectrum, as returned by `cwt` (wavelet.py:123)."""
        return self.engine.signal_fft()

    @_live
    def power(self, rectify=False, variance=None):
        """|W|^2, divided by the scale if `rectify` and by `variance` if given."""
        rs = None
        if rectify or variance is not None:
            rs = np.ones(len(self.scales))
            if rectify:
                rs = rs / np.asarray(self.scales, dtype=float)
            if variance is not None:
                rs = rs / float(variance)
        return self.engine.power(len(self.scales), self.n0, rs)

    def coi_ranges(self):
        """Columns inside the cone of influence, per scale: period_j <= coi[n] holds on one
        centred range [lo_j, hi_j)."""
        return coi_ranges(self.wavelet, self.n0, self.dt, self.period)

    @_live
    def global_power(self, inside_coi=False):
        """Time mean of |W|^2 per scale (`power.mean(axis=1)`); with `inside_coi` only over
        the columns where the period is inside the cone of influence (NaN if there are none)."""
        if not inside_coi:
            return self.engine.global_power(len(self.scales))
        lo, hi = self.coi_ranges()
        return self.engine.global_power_ranges(lo, hi)

    @_live
    def scale_avg_power(self, period_min, period_max, variance=1.0):
        """Scale-averaged power over period_min <= period < period_max (TC98 eq. 24 as in
        simple_sample.py:87-91): variance * dj * dt / Cdelta * sum_j |W_j|^2 / s_j."""
        if self.wavelet.cdelta == -1:
            raise ValueError('Cdelta not defined for this wavelet')
        per = self.period
        sel = (per >= period_min) & (per < period_max)
        w = np.where(sel, 1.0 / np.asarray(self.scales, dtype=float), 0.0)
        w = w * (variance * self.dj * self.dt / self.wavelet.cdelta)
        return self.engine.scale_avg_power(w)

    @_live
    def icwt(self):
        """Inverse transform of the resident coefficients (wavelet.py:169-170)."""
        red = self.engine.icwt_sum()
        fac = self.dj * np.sqrt(self.dt) / (self.wavelet.cdelta * self.wavelet.psi(0))
        if not np.iscomplexobj(fac):
            return fac * red
        # complex factor (Morlet / Paul: psi(0) is complex in the reference, so is its icwt): one pass per
        # component instead of NumPy's promote-then-multiply over N points
        out = self.engine.result_array(red.shape, np.complex128)   # pooled: no first-touch page faults per call
        np.multiply(red, np.real(fac), out=out.real)
        np.multiply(red, np.imag(fac), out=out.imag)
        return out


def cwt_resident(signal, dt, dj=1/12, s0=-1, J=-1, wavelet='morlet', freqs=None, engine=None):
    """Same transform as `cwt` (reference wavelet.py:13-124), W kept on the device.

    Returns a `ResidentTransform`.  Scales whose row the reference would drop as all-NaN
    (Paul at very large scales) are dropped here as well, so `.scales` / `.freqs` equal the
    ones `cwt` returns."""
    wavelet = _check_parameter_wavelet(wavelet)
    spec = wavelet._engine_spec() if hasattr(wavelet, '_engine_spec') else None
    if spec is None:
        # duck-typed objects, subclasses that override psi_ft, non-integer or out-of-range orders
        raise TypeError("cwt_resident needs one of the analytic families the engine evaluates "
                        "itself: Morlet(f0), Paul(m) or DOG(m) with an integer order in [1, 64] "
                        "and the stock psi_ft")
    n0 = len(signal)
    sj, freqs = _resolve_scales(n0, dt, dj, s0, J, wavelet, freqs)
    npad = fft_kwargs(signal)['n']
    keep = ~_nan_rows(wavelet, np.asarray(sj, dtype=float), npad, dt)
    if keep.any():
        sj, freqs = sj[keep], freqs[keep]
    else:
        raise ValueError("every scale of this transform is NaN in the reference")
    eng = engine or _engine.default_engine()
    sig = np.asarray(signal)
    if sig.dtype != np.float32:
        sig = np.asarray(sig, dtype=np.float64)
    family, param = spec
    precision = _precision()
    with eng.lock:
        if _sync_padding(eng, n0):
            precision = _engine.F64
        eng.cwt(sig, dt, sj, family, param, precision, fetch=False)
        serial = eng.job_serial()
    return ResidentTransform(eng, wavelet, n0, dt, dj, sj, freqs, precision, serial)
