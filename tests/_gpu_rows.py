"""Helpers of the row-by-row kernel tests: reference rows, single-row fetches and the kernel
names of a profiled call.  The row gate itself is tests/_rowerr.py."""
import re

import numpy as np
import scipy.fft as sfft

from oracle import cwt_oracle as orc


def oracle_rows(x, sj, rows, mother=None, dt=1.0):
    """Rows `rows` of the reference transform of x (padded to the next power of two) with
    mother wavelet `mother` (default Morlet(6)) and sampling interval dt
    (pycwt/wavelet.py:102-106).  A float32 signal is transformed at its float64 values."""
    mo = mother or orc.Morlet(6)
    x = np.asarray(x, dtype=np.float64)
    n0 = len(x)
    npad = orc.next_pow2(n0)
    xh = sfft.fft(x, npad, workers=-1)
    om = 2 * np.pi * sfft.fftfreq(npad, dt)
    out = np.empty((len(rows), n0), dtype=np.complex128)
    with np.errstate(all="ignore"):
        for i, j in enumerate(rows):
            filt = np.sqrt(sj[j] * om[1] * npad) * np.conj(mo.psi_ft(sj[j] * om))
            out[i] = sfft.ifft(xh * filt, workers=-1)[:n0]
    return out


def fetch_rows(e, rows, n0):
    """Rows of the resident transform, one device-to-host copy each (complex128)."""
    out = np.empty((len(rows), n0), dtype=np.complex128)
    for i, j in enumerate(rows):
        e._check(e.lib.cwtb_get_w(e.h, out[i].ctypes.data, 1, int(j), 1))
    return out


def profiled(e, fn):
    """fn() between profile_begin / profile_end: (its result, the profile).  The profile lists
    every launch in issue order on one stream (the engine's forks are serialised)."""
    e.profile_begin()
    try:
        res = fn()
    finally:
        prof = e.profile_end()
    return res, prof


def kernel_counts(prof, pattern, default=0):
    """{groups of `pattern` matched against each kernel name: launches}.  Numeric groups become
    ints; a group the name does not have (a defaulted template argument) becomes `default`."""
    if isinstance(pattern, str):
        pattern = re.compile(pattern)
    out = {}
    for p in prof:
        m = pattern.search(p["name"])
        if m:
            key = tuple(default if g is None else (int(g) if g.lstrip("-").isdigit() else g)
                        for g in m.groups())
            out[key] = out.get(key, 0) + p["launches"]
    return out
