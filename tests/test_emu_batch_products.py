"""cwt_batch: per-channel products of a batched transform, reduced on the device by
BatchProductsBody (CPU, host-emulation build; see tests/test_emu_kernels.py for what that is).

For every channel, each product must equal (i) the NumPy products of the sample scripts
(pycwt/sample/simple_sample.py:60-91) on the oracle's W and (ii) what `cwt_resident` on the
same engine returns for that channel alone.  The inputs are white-noise channels, cut into
several chunks with a short last one (CWTB_BATCH_MB), so the chunk offsets of the row sums, the
channel factors and the column outputs are all exercised.

The cases are check_* functions that take an engine factory: tests/test_gpu_batch_products.py
runs them on the B200 at config 5's geometry."""
import os

import numpy as np
import pytest

from conftest import ROOT
from oracle import cwt_oracle as orc

# max|got - ref| / max|ref| per channel and product: against the oracle, against per-channel
# cwt_resident on the same engine (the same transform; only the order of the sums differs)
GATES = {"fp64": {"oracle": 1e-12, "resident": 1e-13},
         "fp32": {"oracle": 2e-5, "resident": 1e-6}}

# (public wavelet, oracle mother, dt, dj, s0, J)
CASES = {
    "morlet": (lambda p: p.Morlet(6), orc.Morlet(6), 0.5, 0.25, -1, -1),
    "dog2": (lambda p: p.DOG(2), orc.DOG(2), 0.25, 0.25, -1, -1),
    # rows above s ~ 226 are NaN in the reference (Paul's psi_ft overflows) and are dropped
    "paul4": (lambda p: p.Paul(4), orc.Paul(4), 1.0, 0.25, 2, 36),
    # GPU sizes: config 5's scales (S = 128 at n0 = 2^16), and S = 64 at n0 = 2^18
    "morlet_c5": (lambda p: p.Morlet(6), orc.Morlet(6), 1.0, 1 / 8, 2, 127),
    "morlet_s64": (lambda p: p.Morlet(6), orc.Morlet(6), 1.0, 1 / 4, 2, 63),
}
NCH = 5


@pytest.fixture(scope="module")
def emu_lib():
    from pycwt_b200 import build as _build
    return _build.build_emulation(os.path.join(ROOT, "tests", "_emu"))


def err(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    m = np.max(np.abs(ref))
    if m == 0:
        return 0.0 if np.all(got == 0) else np.inf
    return float(np.max(np.abs(got - ref)) / m)


def white(nch, n0, seed, f32=False):
    X = np.random.RandomState(seed).randn(nch, n0)
    return X.astype(np.float32) if f32 else X


def chunk_mb(n0, S, f32, nch=NCH):
    """CWTB_BATCH_MB that cuts nch channels into chunks of 2..nch-1 (the last one shorter)."""
    per_chan = (8 if f32 else 16) * n0 * S
    mb = max(1, -(-2 * per_chan // (1 << 20)))
    nb = (mb << 20) // per_chan
    assert 2 <= nb < nch and nch % nb, (n0, S, mb, nb)
    return mb


def band_set(period):
    """Disjoint, overlapping, every row, no row."""
    p = np.sort(period)
    return [(p[2], p[6]), (p[10], p[14]), (p[4], p[12]), (0.0, np.inf), (p[0] / 4, p[0] / 3)]


def oracle_products(x, dt, dj, s0, J, mo, bands, var):
    W, sj, freqs, coi, _, _ = orc.cwt(np.asarray(x, dtype=np.float64), dt, dj, s0, J, mo)
    power = np.abs(W) ** 2
    period = 1 / freqs
    inside = period[:, None] <= coi[None, :]
    with np.errstate(invalid="ignore", divide="ignore"):
        glbl_coi = np.where(inside.any(axis=1), (power * inside).sum(axis=1) / inside.sum(axis=1), np.nan)
    rect = power / sj[:, None]
    band = [var * dj * dt / mo.cdelta * rect[(period >= a) & (period < b)].sum(axis=0) for a, b in bands]
    return {"sj": sj, "coi": coi, "period": period, "glbl": power.mean(axis=1), "glbl_coi": glbl_coi,
            "band": band, "icwt": orc.icwt(W, sj, dt, dj, mo)}


def compare_coi(got, ref, what):
    assert np.array_equal(np.isnan(got), np.isnan(ref)), what
    ok = ~np.isnan(ref)
    return err(got[ok], ref[ok])


def check_batch_products(make_engine, monkeypatch, case, n0, prec, nch=NCH, seed=0, mb=None,
                         variance=None, oracle_channels=None):
    """One cwt_batch call with every product; each channel against the oracle and against
    cwt_resident.  Returns the worst errors {(product, against): value}."""
    import pycwt_b200 as pycwt
    wav_f, mo, dt, dj, s0, J = CASES[case]
    wav = wav_f(pycwt)
    f32 = prec == "fp32"
    gate = GATES[prec]
    X = white(nch, n0, seed, f32)
    var = np.linspace(0.5, 2.0, nch) if variance is None else variance
    ref0 = oracle_products(X[0], dt, dj, s0, J, mo, [], 1.0)
    bands = band_set(ref0["period"])
    monkeypatch.setenv("CWTB_PRECISION", prec)
    if mb is None:
        mb = chunk_mb(n0, len(ref0["sj"]), f32, nch)
    monkeypatch.setenv("CWTB_BATCH_MB", str(mb))
    eng = make_engine()
    worst = {}

    def note(key, v, tol):
        worst[key] = max(worst.get(key, 0.0), v)
        assert v <= tol, (case, n0, prec, key, v)

    try:
        r = pycwt.cwt_batch(X, dt, dj, s0, J, wav, inside_coi=True, bands=bands, variance=var,
                            icwt=True, engine=eng)
        assert np.array_equal(r.scales, ref0["sj"]) and np.array_equal(r.coi, ref0["coi"])
        S = len(r.scales)
        assert r.global_power.shape == (nch, S) and r.global_power_coi.shape == (nch, S)
        assert r.scale_avg.shape == (nch, len(bands), n0) and r.icwt.shape == (nch, n0)
        assert np.iscomplexobj(r.icwt) == (not case.startswith("dog"))
        assert not np.isnan(r.global_power).any()
        if case.startswith("morlet"):      # the largest scales lie outside the cone everywhere
            assert np.isnan(r.global_power_coi).any()
        # the band that selects no row is exactly zero
        assert np.all(r.scale_avg[:, -1] == 0)
        # spectra-only call of the engine on the same input
        p_only, _ = eng.cwt_batch(X, dt, r.scales, *wav._engine_spec(), precision=1 if f32 else 0)
        note(("glbl", "cwt_batch"), err(r.global_power, p_only), gate["resident"])
        chans = range(nch) if oracle_channels is None else oracle_channels
        for c in chans:
            ref = oracle_products(X[c], dt, dj, s0, J, mo, bands, var[c])
            note(("glbl", "oracle"), err(r.global_power[c], ref["glbl"]), gate["oracle"])
            note(("glbl_coi", "oracle"), compare_coi(r.global_power_coi[c], ref["glbl_coi"], c), gate["oracle"])
            for b in range(len(bands) - 1):
                note(("band", "oracle"), err(r.scale_avg[c, b], ref["band"][b]), gate["oracle"])
            note(("icwt", "oracle"), err(r.icwt[c], ref["icwt"]), gate["oracle"])
        for c in range(nch):
            res = pycwt.cwt_resident(X[c], dt, dj, s0, J, wav, engine=eng)
            note(("glbl", "resident"), err(r.global_power[c], res.global_power()), gate["resident"])
            note(("glbl_coi", "resident"),
                 compare_coi(r.global_power_coi[c], res.global_power(inside_coi=True), c), gate["resident"])
            for b, (pmin, pmax) in enumerate(bands[:-1]):
                note(("band", "resident"), err(r.scale_avg[c, b], res.scale_avg_power(pmin, pmax, var[c])),
                     gate["resident"])
            note(("icwt", "resident"), err(r.icwt[c], res.icwt()), gate["resident"])
    finally:
        eng.close()
    return worst


def check_products_subsets(make_engine, monkeypatch, n0=1000, prec="fp64"):
    """Products not asked for are None; what is asked for does not depend on the rest."""
    import pycwt_b200 as pycwt
    monkeypatch.setenv("CWTB_PRECISION", prec)
    X = white(3, n0, 7, prec == "fp32")
    eng = make_engine()
    try:
        full = pycwt.cwt_batch(X, 0.5, 0.25, engine=eng, inside_coi=True, bands=[(2, 8)], icwt=True)
        only = pycwt.cwt_batch(X, 0.5, 0.25, engine=eng)
        assert only.global_power_coi is None and only.scale_avg is None and only.icwt is None
        assert err(only.global_power, full.global_power) <= GATES[prec]["resident"]
        ic = pycwt.cwt_batch(X, 0.5, 0.25, engine=eng, icwt=True)
        assert np.array_equal(ic.icwt, full.icwt)
        bd = pycwt.cwt_batch(X, 0.5, 0.25, engine=eng, bands=[(2, 8)], variance=3.0)
        assert err(bd.scale_avg, 3.0 * full.scale_avg) <= GATES[prec]["resident"]
    finally:
        eng.close()


def check_errors(make_engine, monkeypatch):
    import ctypes
    import pycwt_b200 as pycwt
    from pycwt_b200 import _engine, helpers
    eng = make_engine()
    try:
        X = white(3, 256, 1)
        with pytest.raises(ValueError):
            pycwt.cwt_batch(X[0], 1.0, engine=eng)
        with pytest.raises(ValueError):
            pycwt.cwt_batch(np.empty((0, 256)), 1.0, engine=eng)
        with pytest.raises(ValueError):
            pycwt.cwt_batch(X, 1.0, engine=eng, bands=[(2, 8)], variance=[1.0, 2.0])
        with pytest.raises(ValueError):
            pycwt.cwt_batch(X, 1.0, engine=eng, bands=[(2, 3)] * 9)
        with pytest.raises(ValueError):     # every row NaN (Paul far beyond its overflow scale)
            pycwt.cwt_batch(X, 1.0, wavelet=pycwt.Paul(4), freqs=np.array([1e-5, 2e-5]), engine=eng)

        class Duck(object):
            def flambda(self):
                return 1.0

        with pytest.raises(TypeError):
            pycwt.cwt_batch(X, 1.0, wavelet=Duck(), engine=eng)
        helpers.set_fft_padding(False)
        try:
            with pytest.raises(NotImplementedError):
                pycwt.cwt_batch(white(2, 300, 2), 1.0, engine=eng)
            r = pycwt.cwt_batch(X, 1.0, engine=eng)         # a power of two is the same either way
            assert r.global_power.shape == (3, len(r.scales))
        finally:
            helpers.set_fft_padding(True)
            eng.set_padding(True)

        # the C ABI
        lib, h = eng.lib, eng.h
        sj = np.ascontiguousarray(2.0 * 2 ** (np.arange(8) / 4))
        S, n0 = sj.size, X.shape[1]
        P = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
        power = np.empty((3, S))
        pcoi = np.empty((3, S))
        wt = np.ones((9, S))
        band = np.empty((3, 9, n0))
        lo = np.zeros(S, dtype=np.int64)
        hi = np.full(S, n0, dtype=np.int64)
        icw = np.empty((3, n0))

        def call(X=X, n_chan=3, family=0, lo=None, hi=None, nb=0, wt=None, cs=None, want=0,
                 power=power, pcoi=None, band=None, icw=None):
            return lib.cwtb_cwt_batch_products(h, P(X), 0, n_chan, n0, 1.0, P(sj), S, family, 6.0, 0,
                                               P(lo), P(hi), nb, P(wt), P(cs), 1.0, 0.0, want,
                                               P(power), P(pcoi), P(band), P(icw))

        ARG, UNSUP = -1, -5
        assert call() == 0
        assert call(power=None) == ARG
        assert call(X=None) == ARG
        assert call(n_chan=0) == ARG
        assert call(nb=9, wt=wt, band=band) == ARG
        assert call(nb=-1) == ARG
        assert call(nb=2, wt=None, band=band) == ARG
        assert call(nb=2, wt=wt, band=None) == ARG
        assert call(lo=lo, pcoi=pcoi) == ARG
        assert call(hi=hi, pcoi=pcoi) == ARG
        assert call(lo=lo, hi=hi) == ARG                  # ranges without an output
        assert call(want=1) == ARG                        # icwt without an output
        assert call(want=3, icw=icw) == ARG
        assert call(family=_engine.TABLE) == UNSUP
        assert call(lo=lo, hi=hi, pcoi=pcoi, nb=8, wt=wt, band=band, want=1, icw=icw) == 0
        # a NULL chan_scale is 1 for every channel
        cs = np.ones(3)
        b1 = np.empty((3, 2, n0))
        b2 = np.empty((3, 2, n0))
        assert call(nb=2, wt=wt, band=b1) == 0
        assert call(nb=2, wt=wt, band=b2, cs=cs) == 0
        assert np.array_equal(b1, b2)
        eng.set_padding(False)
        try:
            Xo = white(3, 300, 3)
            assert lib.cwtb_cwt_batch_products(h, P(Xo), 0, 3, 300, 1.0, P(sj), S, 0, 6.0, 0, None, None,
                                               0, None, None, 0.0, 0.0, 0, P(power), None, None, None) == UNSUP
        finally:
            eng.set_padding(True)
    finally:
        eng.close()


# ---- the emulation runs ----------------------------------------------------------------------
def _factory(emu_lib):
    from pycwt_b200 import _engine
    return lambda: _engine.Engine(0, lib_path=emu_lib)


@pytest.mark.parametrize("n0", [1000, 3001, 4096])
def test_morlet_fp64(emu_lib, monkeypatch, n0):
    w = check_batch_products(_factory(emu_lib), monkeypatch, "morlet", n0, "fp64", seed=n0)
    print("morlet fp64 n0=%d:" % n0, {k: "%.1e" % v for k, v in w.items()})


@pytest.mark.parametrize("n0", [1000, 4096])
def test_morlet_fp32(emu_lib, monkeypatch, n0):
    w = check_batch_products(_factory(emu_lib), monkeypatch, "morlet", n0, "fp32", seed=n0 + 1)
    print("morlet fp32 n0=%d:" % n0, {k: "%.1e" % v for k, v in w.items()})


def test_dog2_real_icwt(emu_lib, monkeypatch):
    w = check_batch_products(_factory(emu_lib), monkeypatch, "dog2", 3001, "fp64", seed=5)
    print("dog2 fp64:", {k: "%.1e" % v for k, v in w.items()})


def test_paul4_dropped_rows(emu_lib, monkeypatch):
    import pycwt_b200 as pycwt
    sj, _ = pycwt.batch._resolve_scales(1000, 1.0, 0.25, 2, 36, pycwt.Paul(4), None)
    assert len(sj) == 37 and sj.max() > 226          # some rows will be dropped
    w = check_batch_products(_factory(emu_lib), monkeypatch, "paul4", 1000, "fp64", seed=6)
    print("paul4 fp64:", {k: "%.1e" % v for k, v in w.items()})


def test_scalar_variance_one_chunk(emu_lib, monkeypatch):
    check_batch_products(_factory(emu_lib), monkeypatch, "morlet", 1000, "fp64", seed=8, mb=64,
                         variance=np.full(NCH, 1.0))


def test_products_subsets(emu_lib, monkeypatch):
    check_products_subsets(_factory(emu_lib), monkeypatch)


def test_errors(emu_lib, monkeypatch):
    check_errors(_factory(emu_lib), monkeypatch)


def test_coi_ranges_unchanged():
    """The module-level COI ranges equal the closed form they replace in ResidentTransform."""
    import pycwt_b200 as pycwt
    from pycwt_b200.resident import coi_ranges
    for wav, n0, dt in [(pycwt.Morlet(6), 1000, 0.5), (pycwt.Paul(4), 3001, 1.0), (pycwt.DOG(2), 4096, 0.25)]:
        sj, freqs = pycwt.batch._resolve_scales(n0, dt, 0.25, -1, -1, wav, None)
        period = 1 / freqs
        lo, hi = coi_ranges(wav, n0, dt, period)
        c = wav.flambda() * wav.coi() * dt
        coi = c * (n0 / 2 - np.abs(np.arange(n0) - (n0 - 1) / 2))
        inside = period[:, None] <= coi[None, :]
        for j in range(len(period)):
            cols = np.flatnonzero(inside[j])
            if cols.size:
                assert (lo[j], hi[j]) == (cols[0], cols[-1] + 1)
            else:
                assert lo[j] == hi[j]
