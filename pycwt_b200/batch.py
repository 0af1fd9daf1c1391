"""Batched transform of many channels with per-channel products reduced on the device.

Sensor arrays, EEG/MEG montages and climate grids are many series of one length.  `cwt_batch`
transforms them together (channels of a chunk share every kernel launch) and returns, per
channel, the products the reference's sample scripts build from W
(pycwt/sample/simple_sample.py:60-96) -- never W itself, which at 1024 channels of 2^16 samples
is 512 GiB:

    global_power      power.mean(axis=1)                                   (:79)
    global_power_coi  the same mean over the columns inside the cone of influence
    scale_avg         variance * dj*dt/Cdelta * sum_{j in band} power[j] / s_j   (:88-91)
    icwt              icwt(W, ...)                                         (:60)

One kernel per chunk reads every coefficient once while the chunk is resident in HBM; only
O(C*S) and O(C*n0) numbers cross the bus.  For each channel the results equal those of
`cwt_resident(X[c], ...)` and its `.global_power()`, `.global_power(inside_coi=True)`,
`.scale_avg_power(pmin, pmax, variance[c])` and `.icwt()`.
"""
import collections

import numpy as np

from . import _engine
from .helpers import fft_kwargs
from .resident import coi_curve, coi_ranges
from .wavelet import _check_parameter_wavelet, _nan_rows, _precision, _resolve_scales, _sync_padding

__all__ = ['cwt_batch', 'BatchProducts']

MAX_BANDS = 8

BatchProducts = collections.namedtuple(
    'BatchProducts', ['scales', 'freqs', 'coi', 'global_power', 'global_power_coi', 'scale_avg', 'icwt'])
BatchProducts.__doc__ = """Per-channel products of `cwt_batch` (None where not requested).

    scales, freqs     [S]        the scales kept (rows the reference drops as NaN are dropped)
    coi               [n0]       cone of influence, as `cwt` returns it
    global_power      [C, S]     time mean of |W|^2
    global_power_coi  [C, S]     the same inside the cone of influence (NaN where it is empty)
    scale_avg         [C, B, n0] scale-averaged power of each band
    icwt              [C, n0]    inverse transform (complex for Morlet and Paul, real for DOG)"""


def cwt_batch(X, dt, dj=1/12, s0=-1, J=-1, wavelet='morlet', freqs=None, *,
              inside_coi=False, bands=(), variance=1.0, icwt=False, engine=None):
    """Transform every row of X [channels, samples] and reduce each channel's coefficients on
    the device.  Scales follow `cwt` (dj, s0, J, wavelet, freqs).

    inside_coi  also return the global spectrum restricted to the cone of influence;
    bands       (period_min, period_max) pairs, at most 8: scale-averaged power over
                period_min <= period < period_max, per channel;
    variance    scalar or one value per channel: factor of the scale-averaged power;
    icwt        also return the inverse transform of every channel.

    Returns a `BatchProducts`.  The arithmetic follows CWTB_PRECISION like every other call."""
    wavelet = _check_parameter_wavelet(wavelet)
    spec = wavelet._engine_spec() if hasattr(wavelet, '_engine_spec') else None
    if spec is None:
        raise TypeError("cwt_batch needs one of the analytic families the engine evaluates "
                        "itself: Morlet(f0), Paul(m) or DOG(m) with an integer order in [1, 64] "
                        "and the stock psi_ft")
    X = np.asarray(X)
    if X.ndim != 2 or X.size == 0:
        raise ValueError("cwt_batch: X must be a non-empty 2-D array [channels, samples]")
    if X.dtype != np.float32:
        X = np.asarray(X, dtype=np.float64)
    nch, n0 = X.shape
    bands = [tuple(float(p) for p in b) for b in bands]
    if len(bands) > MAX_BANDS:
        raise ValueError("cwt_batch: at most %d bands" % MAX_BANDS)
    if any(len(b) != 2 for b in bands):
        raise ValueError("cwt_batch: each band is a (period_min, period_max) pair")
    var = np.asarray(variance, dtype=np.float64)
    if var.ndim == 0:
        var = np.full(nch, float(var))
    elif var.shape != (nch,):
        raise ValueError("cwt_batch: variance must be a scalar or one value per channel "
                         "(%d), got shape %s" % (nch, var.shape))
    if bands and wavelet.cdelta == -1:
        raise ValueError('Cdelta not defined for this wavelet')

    sj, freqs = _resolve_scales(n0, dt, dj, s0, J, wavelet, freqs)
    eng = engine or _engine.default_engine()
    family, param = spec
    precision = _precision()
    with eng.lock:
        if _sync_padding(eng, n0):
            raise NotImplementedError("cwt_batch runs padded transforms only: with the un-padded "
                                      "length policy, n0 must be a power of two (transform "
                                      "channels one at a time with cwt)")
        npad = fft_kwargs(range(n0))['n']      # transform length (helpers.py:15-30)
        keep = ~_nan_rows(wavelet, np.asarray(sj, dtype=float), npad, dt)
        if not keep.any():
            raise ValueError("every scale of this transform is NaN in the reference")
        sj, freqs = sj[keep], freqs[keep]
        period = 1.0 / np.asarray(freqs)
        rng = coi_ranges(wavelet, n0, dt, period) if inside_coi else None
        wt = None
        if bands:
            inv_s = 1.0 / np.asarray(sj, dtype=float)
            wt = np.stack([np.where((period >= pmin) & (period < pmax), inv_s, 0.0)
                           * (dj * dt / wavelet.cdelta) for pmin, pmax in bands])
        fac = dj * np.sqrt(dt) / (wavelet.cdelta * wavelet.psi(0)) if icwt else None
        power, power_coi, band, iw = eng.cwt_batch_products(
            X, dt, sj, family, param, precision, coi_ranges=rng, band_weights=wt,
            chan_scale=var if bands else None, icwt_factor=fac)
    return BatchProducts(sj, freqs, coi_curve(wavelet, n0, dt), power, power_coi, band, iw)
