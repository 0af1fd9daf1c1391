"""CPU-only logic tests of the CUDA kernel bodies through the host-emulation build.

tests/_emu/libcwtb200_emu.so is the SAME kernel source compiled with -DCWTB_HOST_EMU, where
every CTA runs as a plain C++ loop over (phase, thread).  It exists so that index maths,
plans, pruning and epilogues can be checked where no GPU is present (the build container).
It is test infrastructure only: the package never loads it (pycwt_b200._engine.LIB_PATH is the
sm_100a library) and these tests patch the loader path only for their own duration."""
import numpy as np
import pytest

from conftest import ROOT, load_golden, relerr, golden_cwt_kwargs
from _rowerr import check_rows
from oracle import cwt_oracle as orc


@pytest.fixture(scope="module")
def emu():
    import os
    from pycwt_b200 import build as _build, _engine
    lib = _build.build_emulation(os.path.join(ROOT, "tests", "_emu"))
    eng = _engine.Engine(0, lib_path=lib)
    assert "emulation" in eng.version()
    yield eng
    eng.close()


def test_fft_plans_all_lengths(emu):
    rs = np.random.RandomState(0)
    for n in [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 8192]:
        x = rs.randn(2, n) + 1j * rs.randn(2, n)
        assert relerr(emu.fft_c2c(x, -1), np.fft.fft(x, axis=1)) < 1e-13
        assert relerr(emu.fft_c2c(x, +1, precision=1), np.fft.ifft(x, axis=1) * n) < 5e-6


@pytest.mark.parametrize("name", ["nino3_morlet_tutorial", "nino3_paul_default", "nino3_dog3_odd",
                                  "chirp4000_morlet"])
def test_cwt_kernels_vs_reference_fixture(emu, name):
    g = load_golden(name)
    fam = {"morlet": 0, "paul": 1, "dog": 2}[str(g["wavelet"])]
    W = emu.cwt(g["x"], float(g["dt"]), g["sj"], fam, float(g["param"]))
    st = int(g["stride"])
    assert relerr(W[:, ::st], g["W"]) < 1e-10


def test_every_pruned_class_and_dense_path(emu):
    """Exact mode (expansion off): every pruned length 2^5..2^15 and the dense path, every row
    on its own (tests/test_emu_exact.py: the row gates of the exact path), on a chirp in white
    noise and on white noise alone."""
    from test_emu_exact import GATE
    n = 2 ** 15
    t = np.arange(n) / n
    noise = np.random.RandomState(1).randn(n)
    sj = 2.0 * 2 ** (np.arange(0, 27) / 2.0)
    m = orc.Morlet(6)
    emu.set_expand_eps(0.0, 0.0)
    try:
        for x in (np.sin(2 * np.pi * (50 * t + (n / 8) * t ** 2)) + 0.1 * noise, noise):
            Wr = orc.cwt(x, 1.0, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
            W = emu.cwt(x, 1.0, sj, 0, 6.0)
            plan = emu.last_plan(len(sj))
            assert set(plan) >= set(range(5, 16)), plan   # single, direct (11..13), two-kernel, dense
            err = check_rows(W, Wr, *GATE[0], what="fp64")
            W32 = emu.cwt(x.astype(np.float32), 1.0, sj, 0, 6.0, precision=1)
            Wr32 = orc.cwt(x.astype(np.float32).astype(np.float64), 1.0, wavelet=m,
                           freqs=1 / (m.flambda() * sj))[0]
            err32 = check_rows(W32, Wr32, *GATE[1], what="fp32")
            print("exact rows: worst row error fp64 %.2e, fp32 %.2e" % (err, err32))
    finally:
        emu.set_expand_eps()


def test_expansion_path_every_coarse_length(emu):
    """Default mode: scales whose band is <= 1/32 of the transform length run as coarse transform +
    polyphase Kaiser-Bessel expansion (kernels.cuh: ExpandBody); every family, fp64 and fp32,
    including the cross-product epilogue.  The alias bound is 5e-13; measured ~1e-14."""
    n = 2 ** 15
    t = np.arange(n) / n
    x = np.sin(2 * np.pi * (50 * t + (n / 8) * t ** 2)) + 0.1 * np.random.RandomState(1).randn(n)
    sj = 2.0 * 2 ** (np.arange(0, 27) / 2.0)
    for fam, ref, par, s in ((0, orc.Morlet(6), 6.0, sj), (1, orc.Paul(4), 4.0, sj[:14]),
                             (2, orc.DOG(2), 2.0, sj), (2, orc.DOG(3), 3.0, sj)):
        Wr = orc.cwt(x, 1.0, wavelet=ref, freqs=1 / (ref.flambda() * s))[0]
        W = emu.cwt(x, 1.0, s, fam, par)
        plan = emu.last_plan(len(s))
        assert min(plan) < 0 and max(plan) == 15 or fam == 1, plan
        assert relerr(W, Wr) < 2e-13, (fam, relerr(W, Wr))
        # every expansion row on its own (the global maximum hides the small rows)
        rows = [i for i, p in enumerate(plan) if p < 0]
        assert rows
        err = check_rows(W[rows], Wr[rows], 1e-12, 1e-14, what=fam)
        print("family %d: worst expansion row error %.2e" % (fam, err))
        W32 = emu.cwt(x.astype(np.float32), 1.0, s, fam, par, precision=1)
        assert min(emu.last_plan(len(s))) < 0
        assert relerr(W32, Wr) < 1e-5
    # Morlet: coarse lengths 2^6 .. 2^12 all occur
    emu.cwt(x, 1.0, sj, 0, 6.0)
    assert set(emu.last_plan(len(sj))) >= set(range(-12, -5)), emu.last_plan(len(sj))
    # odd length (trimmed output), cross-product epilogue on expansion rows
    rs = np.random.RandomState(5)
    y1, y2 = rs.randn(5001), rs.randn(5001)
    s2 = 2.0 * 2 ** (np.arange(0, 20) / 2.0)
    m = orc.Morlet(6)
    W1 = orc.cwt(y1, 1.0, wavelet=m, freqs=1 / (m.flambda() * s2))[0]
    W2 = orc.cwt(y2, 1.0, wavelet=m, freqs=1 / (m.flambda() * s2))[0]
    assert relerr(emu.xwt(y1, y2, 1.0, s2, 0, 6.0), W1 * np.conj(W2)) < 2e-13
    assert min(emu.last_plan(len(s2))) < 0


def test_xwt_wct_smooth_kernels(emu):
    g = load_golden("ao_baltic_xwt_wct")
    y1 = (g["y1"] - g["y1"].mean()) / g["y1"].std()
    y2 = (g["y2"] - g["y2"].mean()) / g["y2"].std()
    m = orc.Morlet(6)
    sj = 2 * float(g["dt"]) / m.flambda() * 2 ** (np.arange(76) / 12.0)
    assert relerr(emu.xwt(y1, y2, float(g["dt"]), sj, 0, 6.0), g["W12"]) < 1e-10
    WCT, aWCT = emu.wct(y1, y2, float(g["dt"]), 1 / 12, sj, 0, 6.0, 14)
    assert relerr(WCT, g["WCT"]) < 1e-10 and relerr(aWCT, g["aWCT"]) < 1e-10
    s = load_golden("smooth_cases")
    assert relerr(emu.smooth(s["Wc"], 1.0, s["sj"], 5), s["Sc"]) < 1e-10
    assert relerr(emu.smooth(s["Wr"], 1.0, s["sj"], 5), s["Sr"]) < 1e-10


def test_batched_rows_equal_single_channel(emu):
    rs = np.random.RandomState(3)
    X = rs.randn(3, 5000)
    sj = 2.0 * 2 ** (np.arange(0, 20) / 2.0)
    power, W = emu.cwt_batch(X, 1.0, sj, 0, 6.0, want_w=True)
    for ch in range(3):
        assert np.array_equal(W[ch], emu.cwt(X[ch], 1.0, sj, 0, 6.0))


def test_error_paths_report_status_and_message(emu):
    """The C ABI never throws: bad calls return a negative status + message, which the
    ctypes layer turns into EngineError."""
    from pycwt_b200._engine import EngineError
    x = np.random.RandomState(0).randn(64)
    with pytest.raises(EngineError, match="family"):
        emu.cwt(x, 1.0, np.array([2.0, 4.0]), 7, 6.0)
    with pytest.raises(EngineError, match="order"):
        emu.cwt(x, 1.0, np.array([2.0, 4.0]), 1, 2.5)          # Paul order must be an integer
    with pytest.raises(EngineError, match="dt"):
        emu.cwt(x, -1.0, np.array([2.0]), 0, 6.0)
    with pytest.raises(EngineError, match="table"):
        emu.cwt(x, 1.0, np.array([2.0]), 3, 0.0)                # CWTB_TABLE without a table
    with pytest.raises(EngineError):
        emu.set_band_eps(0.5)
    with pytest.raises(ValueError):
        emu.xwt(np.zeros(10), np.zeros(11), 1.0, np.array([2.0]), 0, 6.0)
    # a failed call leaves the context usable
    W = emu.cwt(x, 1.0, np.array([2.0, 4.0]), 0, 6.0)
    assert W.shape == (2, 64) and np.isfinite(W).all()


def test_table_family_matches_analytic(emu):
    """CWTB_TABLE (duck-typed wavelets: host-evaluated response) == analytic Morlet path."""
    rs = np.random.RandomState(2)
    for n0 in (300, 3000):
        x = rs.randn(n0)
        sj = 2.0 * 2 ** (np.arange(12) / 2.0)
        npad = orc.next_pow2(n0)
        om = 2 * np.pi * np.fft.fftfreq(npad, 1.0)
        table = (sj[:, None] * om[1] * npad) ** .5 * np.conj(orc.Morlet(6).psi_ft(sj[:, None] * om))
        Wt = emu.cwt(x, 1.0, sj, 3, 0.0, table=table)
        Wa = emu.cwt(x, 1.0, sj, 0, 6.0)
        assert relerr(Wt, Wa) < 1e-13


def test_three_level_path_beyond_2_20(emu):
    """Np = 2^21: pre-pass + interleaved 2^20-point transforms (forward FFT and dense scales),
    pruned classes unchanged."""
    rs = np.random.RandomState(4)
    y = rs.randn(1, 2 ** 21) + 1j * rs.randn(1, 2 ** 21)
    assert relerr(emu.fft_c2c(y, -1), np.fft.fft(y, axis=1)) < 1e-13
    n0 = 2 ** 20 + 777
    x = rs.randn(n0)
    sj = np.array([2.0, 7.0, 300.0, 5e4])
    W = emu.cwt(x, 1.0, sj, 0, 6.0)
    assert emu.last_plan(4)[0] == 21
    m = orc.Morlet(6)
    Wr = orc.cwt(x, 1.0, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
    assert relerr(W, Wr) < 1e-10


def _sample_products(x, dt, dj, s0, J, mother_o):
    """The derived products of pycwt/sample/simple_sample.py:64-91 in NumPy on the oracle's W."""
    W, sj, freqs, coi, _, _ = orc.cwt(x, dt, dj, s0, J, mother_o)
    power = np.abs(W) ** 2
    period = 1 / freqs
    out = {"W": W, "sj": sj, "power": power, "rect": power / sj[:, None],
           "glbl": power.mean(axis=1), "coi": coi, "period": period}
    sel = (period >= 2) & (period < 8)
    out["scale_avg"] = 1.7 * dj * dt / mother_o.cdelta * (power / sj[:, None])[sel].sum(axis=0)
    inside = period[:, None] <= coi[None, :]
    with np.errstate(invalid="ignore", divide="ignore"):
        out["glbl_coi"] = np.where(inside.any(axis=1), (power * inside).sum(axis=1) / inside.sum(axis=1), np.nan)
    out["iW"] = orc.icwt(W, sj, dt, dj, mother_o)
    return out


def check_resident_products(eng, precision_tol=1e-12):
    import pycwt_b200 as pycwt
    g = load_golden("nino3_morlet_tutorial")
    x, dt = g["x"], float(g["dt"])
    ref = _sample_products(x, dt, 0.25, 0.5, 28, orc.Morlet(6))
    r = pycwt.cwt_resident(x, dt, 0.25, 0.5, 28, pycwt.Morlet(6), engine=eng)
    assert r.shape == ref["W"].shape
    assert np.array_equal(r.scales, ref["sj"]) and np.array_equal(r.coi, ref["coi"])
    assert relerr(r.power(), ref["power"]) < precision_tol
    assert relerr(r.power(rectify=True), ref["rect"]) < precision_tol
    assert relerr(r.power(variance=2.5), ref["power"] / 2.5) < precision_tol
    assert relerr(r.global_power(), ref["glbl"]) < precision_tol
    got = r.global_power(inside_coi=True)
    assert np.array_equal(np.isnan(got), np.isnan(ref["glbl_coi"])) and np.isnan(got).any()
    ok = ~np.isnan(got)
    assert relerr(got[ok], ref["glbl_coi"][ok]) < precision_tol
    assert relerr(r.scale_avg_power(2, 8, variance=1.7), ref["scale_avg"]) < precision_tol
    assert relerr(r.icwt(), ref["iW"]) < precision_tol
    assert relerr(r.wave(), ref["W"]) < precision_tol
    # the handle dies with the next transform on the same engine
    eng.cwt(x, dt, ref["sj"][:3], 0, 6.0, fetch=False)
    with pytest.raises(pycwt.EngineError):
        r.global_power()


def test_resident_transform_products(emu):
    check_resident_products(emu)


def test_dft_of_any_length(emu):
    """cwtb_fft_c2c for lengths that are not powers of two (Bluestein on the 2^k kernels)."""
    rs = np.random.RandomState(3)
    for n in [3, 5, 6, 7, 12, 100, 147, 504, 1000, 1023, 1025, 4001]:
        x = rs.randn(2, n) + 1j * rs.randn(2, n)
        assert relerr(emu.fft_c2c(x, -1), np.fft.fft(x, axis=1)) < 1e-13, n
        assert relerr(emu.fft_c2c(x, +1), np.fft.ifft(x, axis=1) * n) < 1e-13, n


def check_unpadded_mode(eng, tol):
    """Un-padded transforms (the reference's pyfftw length policy) through the public API
    against fixtures made by the reference's own code with that policy."""
    import pycwt_b200 as pycwt
    from pycwt_b200 import helpers
    helpers.set_fft_padding(False)
    try:
        for name in ["nopad_nino3_morlet", "nopad_nino3_paul", "nopad_nino501_paul", "nopad_nino3_dog3",
                     "nopad_chirp4001_morlet", "nopad_chirp3000_dog"]:
            g = load_golden(name)
            cls = {"morlet": pycwt.Morlet, "paul": pycwt.Paul, "dog": pycwt.DOG}[str(g["wavelet"])]
            mother = cls(int(g["param"]))
            kw = golden_cwt_kwargs(g)
            W, sj, freqs, coi, fft, fftfreqs = pycwt.cwt(g["x"], float(g["dt"]), wavelet=mother, **kw)
            assert tuple(W.shape) == tuple(g["shape"]), name
            st = int(g["stride"])
            assert relerr(W[:, ::st], g["W"]) < tol, (name, relerr(W[:, ::st], g["W"]))
            assert np.array_equal(sj, g["sj"]) and np.array_equal(freqs, g["freqs"])
            assert relerr(fft, g["fft"]) < tol and np.array_equal(fftfreqs, g["fftfreqs"])
            np.testing.assert_allclose(coi, g["coi"], rtol=1e-15)
            if "iW" in g.files:
                iW = pycwt.icwt(W, sj, float(g["dt"]), kw.get("dj", 1 / 12), mother)
                assert relerr(iW, g["iW"]) < tol
        g = load_golden("nopad_ao_baltic_xwt")
        W12, coi, freq, signif = pycwt.xwt(g["y1"], g["y2"], float(g["dt"]), dj=1 / 12,
                                           wavelet=pycwt.Morlet(6))
        assert relerr(W12, g["W12"]) < tol
        np.testing.assert_allclose(signif, g["signif"], rtol=1e-12)
        # duck-typed wavelet (host table) and the device-resident handle follow the same policy
        class Duck(object):
            def __init__(self):
                self.m = pycwt.Morlet(6)
            def __getattr__(self, k):
                if k == '_engine_spec':
                    raise AttributeError(k)
                return getattr(self.m, k)
        g = load_golden("nopad_nino3_morlet")
        Wd = pycwt.cwt(g["x"], 0.25, 0.25, 0.5, 28, Duck())[0]
        assert relerr(Wd, g["W"]) < tol
        r = pycwt.cwt_resident(g["x"], 0.25, 0.25, 0.5, 28, pycwt.Morlet(6))
        assert r.npad == 504 and relerr(r.global_power(), (np.abs(g["W"]) ** 2).mean(axis=1)) < tol
        # coherence, smoothing and the Monte-Carlo levels: the Gaussian filter is circular at the
        # rows' own length in this mode
        g = load_golden("nopad_wct_smooth")
        m = pycwt.Morlet(6)
        assert relerr(m.smooth(g["Wr"], 1.0, 0.25, g["sj"]), g["Sr"]) < tol
        assert relerr(m.smooth(g["Wc"], 1.0, 0.25, g["sj"]), g["Sc"]) < tol
        WCT, aWCT, _, _, _ = pycwt.wct(g["y1"], g["y2"], float(g["dt"]), dj=1 / 12, sig=False, wavelet=m)
        assert relerr(WCT, g["WCT"]) < 100 * tol and relerr(aWCT, g["aWCT"]) < 100 * tol
        np.random.seed(4321)
        sig95 = pycwt.wct_significance(0.2, 0.1, 1.0, 0.5, 2.0, 10, 0.95, m, mc_count=5,
                                       progress=False, cache=False)
        np.testing.assert_allclose(sig95, g["sig95"], rtol=1e-9, equal_nan=True)
    finally:
        helpers.set_fft_padding(True)
    # back in the padded mode the same call gives the padded result again
    g = load_golden("nino3_morlet_tutorial")
    W = pycwt.cwt(g["x"], 0.25, 0.25, 0.5, 28, pycwt.Morlet(6))[0]
    assert relerr(W, g["W"]) < tol


def test_unpadded_mode_public_api(emu, monkeypatch):
    from pycwt_b200 import _engine
    monkeypatch.setattr(_engine, "default_engine", lambda *a, **k: emu)
    check_unpadded_mode(emu, 1e-12)


def test_python_side_shape_guards(emu):
    """The C side sizes its copies from the resident job; the ctypes layer refuses calls whose
    array shapes disagree with it instead of letting them overrun."""
    x = np.random.RandomState(0).randn(100)
    sj = np.array([2.0, 4.0, 8.0])
    emu.cwt(x, 1.0, sj, 0, 6.0, fetch=False)
    with pytest.raises(ValueError):
        emu.get_w(3, 64)                 # wrong column count
    with pytest.raises(ValueError):
        emu.get_w(4, 100)                # more rows than resident
    with pytest.raises(ValueError):
        emu.global_power(5)
    with pytest.raises(ValueError):
        emu.power(3, 99)
    with pytest.raises(ValueError):
        emu.scale_avg_power(np.ones(2))
    with pytest.raises(ValueError):
        emu.global_power_ranges(np.zeros(3), np.ones(4))
    with pytest.raises(ValueError):
        emu.smooth(np.ones((4, 100)), 1.0, sj, 5)
    assert emu.get_w(2, 100).shape == (2, 100) and emu.global_power(3).shape == (3,)


def check_seeded_monte_carlo(eng):
    """Seeded (device-RNG) mode of the Monte-Carlo significance: the Philox surrogates are standard
    normal white noise, a pure function of (seed, pair number); the histograms do not depend on how
    the pairs are split over calls; the significance levels agree with the host-RNG mode within
    the Monte-Carlo scatter."""
    import pycwt_b200 as pycwt
    from pycwt_b200 import wavelet as wv
    z = eng.mc_surrogates(7, 3, 2, 20001)                  # pairs 3 and 4, odd length
    assert z.shape == (2, 2, 20001) and np.isfinite(z).all()
    flat = z.ravel()
    assert abs(flat.mean()) < 4 / np.sqrt(flat.size) and abs(flat.std() - 1) < 0.02
    assert abs(((flat[:-1] * flat[1:]).mean())) < 4 / np.sqrt(flat.size)       # white
    assert abs((flat ** 4).mean() - 3) < 0.15 and np.abs(flat).max() < 7        # Gaussian tails
    assert np.array_equal(eng.mc_surrogates(7, 4, 1, 20001)[0], z[1])          # keyed by pair number
    assert not np.array_equal(eng.mc_surrogates(8, 3, 1, 20001)[0], z[0])      # and by seed
    assert abs(np.corrcoef(z[0, 0], z[0, 1])[0, 1]) < 0.05                      # the two series differ
    m = pycwt.Morlet(6)
    dt, dj, s0, J = 1.0, 0.5, 2.0, 8
    prob = wv._mc_problem(dt, dj, s0, J, m)
    h_all = wv._mc_histogram_seeded(prob, dt, dj, m, 11, 0, 6, engine=eng)
    h_split = (wv._mc_histogram_seeded(prob, dt, dj, m, 11, 0, 2, engine=eng) +
               wv._mc_histogram_seeded(prob, dt, dj, m, 11, 2, 4, engine=eng))
    assert np.array_equal(h_all, h_split) and h_all.sum() > 0
    # against the host-RNG mode (numpy stream): same distribution, different draws
    rs = np.random.RandomState(3)
    tau = int(np.ceil(-2 / np.log(0.3)))
    h_host = wv._mc_histogram(prob, dt, dj, m, lambda i: (rs.randn(prob['N'] + tau)[tau:], rs.randn(prob['N'] + tau)[tau:]),
                              range(40), engine=eng)
    h_dev = wv._mc_histogram_seeded(prob, dt, dj, m, 5, 0, 40, engine=eng)
    a, b = wv._mc_levels(prob, h_host, 0.95), wv._mc_levels(prob, h_dev, 0.95)
    ok = np.isfinite(a)
    assert (np.isfinite(b) == ok).all()
    # the 95 % level of R^2 from 40 pairs: independent runs scatter by ~0.01 at the small scales
    # (many independent samples per row) and by several 0.01 at the largest ones (few)
    d = np.abs(a[ok] - b[ok])
    assert d[:4].max() < 0.03 and d.max() < 0.15, d


def test_seeded_monte_carlo(emu):
    check_seeded_monte_carlo(emu)


def check_generic_smoothing(eng_patch_api):
    """Opt-in smoothing for Paul / DOG (SURVEY 8f rank 4): off by default (`wct` raises AttributeError
    like the reference); when enabled, `smooth` and `wct(sig=False)` match the independent NumPy
    statement of the same definition (oracle.smooth_generic)."""
    pycwt = eng_patch_api
    from pycwt_b200 import mothers
    rs = np.random.RandomState(21)
    n = 700
    y1 = rs.randn(n).cumsum() * 0.1 + rs.randn(n)
    y2 = 0.5 * y1 + rs.randn(n)
    dt, dj = 0.5, 0.25
    with pytest.raises(AttributeError):
        pycwt.wct(y1, y2, dt, dj, sig=False, wavelet=pycwt.Paul(4))
    old = mothers.enable_generic_smoothing(True)
    try:
        for mo, mr in ((pycwt.Paul(4), orc.Paul(4)), (pycwt.DOG(2), orc.DOG(2)), (pycwt.DOG(6), orc.DOG(6))):
            Wc = rs.randn(9, 300) + 1j * rs.randn(9, 300)
            sj = 1.0 * 2 ** (np.arange(9) * dj)
            ref = orc.smooth_generic(Wc, dt, dj, sj, mr)
            assert relerr(mo.smooth(Wc, dt, dj, sj), ref) < 1e-10
            refr = orc.smooth_generic(np.abs(Wc) ** 2, dt, dj, sj, mr)
            got = mo.smooth(np.abs(Wc) ** 2, dt, dj, sj)
            assert not np.iscomplexobj(got) and relerr(got, refr) < 1e-10
            # coherence with this operator: oracle pipeline (wavelet.py:498-514) with the generic smooth
            WCT, aWCT, coi, freq, sig = pycwt.wct(y1, y2, dt, dj, s0=2 * dt, J=20, sig=False, wavelet=mo)
            y1n, y2n = (y1 - y1.mean()) / y1.std(), (y2 - y2.mean()) / y2.std()
            W1, s, *_ = orc.cwt(y1n, dt, dj, 2 * dt, 20, mr)
            W2 = orc.cwt(y2n, dt, dj, 2 * dt, 20, mr)[0]
            inv = 1.0 / s[:, None]
            S1 = orc.smooth_generic(np.abs(W1) ** 2 * inv, dt, dj, s, mr)
            S2 = orc.smooth_generic(np.abs(W2) ** 2 * inv, dt, dj, s, mr)
            S12 = orc.smooth_generic(W1 * W2.conj() * inv, dt, dj, s, mr)
            assert relerr(WCT, np.abs(S12) ** 2 / (S1 * S2)) < 1e-9, type(mo).__name__
        with pytest.raises(ValueError):          # no deltaj0 tabulated for this order
            pycwt.wct(y1, y2, dt, dj, sig=False, wavelet=pycwt.Paul(3))
    finally:
        mothers.enable_generic_smoothing(old)
    # Morlet keeps the reference's Gaussian whatever the switch
    assert hasattr(pycwt.Morlet(6), "smooth")


def test_generic_smoothing_for_paul_and_dog(emu):
    import pycwt_b200 as pycwt
    from pycwt_b200 import _engine
    saved = _engine.default_engine
    _engine.default_engine = lambda *a, **k: emu
    try:
        check_generic_smoothing(pycwt)
    finally:
        _engine.default_engine = saved


def test_plan_reuse_and_invalidation(emu):
    """A call with the geometry of the resident plan reuses it (no re-planning, no descriptor
    upload); any change of geometry or tolerance builds a new one.  Results must not depend on
    which of the two happened."""
    rs = np.random.RandomState(12)
    n = 3000
    sj = 2.0 * 2 ** (np.arange(30) / 4.0)
    m = orc.Morlet(6)

    def ref(x, s):
        return orc.cwt(x, 1.0, wavelet=m, freqs=1 / (m.flambda() * s))[0]

    x1, x2 = rs.randn(n), rs.randn(n).cumsum()
    W1 = emu.cwt(x1, 1.0, sj, 0, 6.0)
    p1 = emu.last_plan(len(sj))
    W2 = emu.cwt(x2, 1.0, sj, 0, 6.0)                    # same plan, other signal
    assert emu.last_plan(len(sj)) == p1
    assert relerr(W1, ref(x1, sj)) < 1e-10 and relerr(W2, ref(x2, sj)) < 1e-10
    W3 = emu.cwt(x2, 1.0, sj[::-1].copy(), 0, 6.0)       # same values, other order: a different plan
    assert relerr(W3, ref(x2, sj[::-1])) < 1e-10
    W4 = emu.cwt(x2[:2999], 1.0, sj, 0, 6.0)             # other length
    assert W4.shape == (30, 2999) and relerr(W4, ref(x2[:2999], sj)) < 1e-10
    emu.set_expand_eps(0.0, 0.0)                          # same geometry, expansion off: must re-plan
    try:
        W5 = emu.cwt(x2[:2999], 1.0, sj, 0, 6.0)
        assert min(emu.last_plan(len(sj))) > 0
    finally:
        emu.set_expand_eps()
    assert relerr(W5, ref(x2[:2999], sj)) < 1e-10
    W6 = emu.cwt(x2[:2999], 1.0, sj, 0, 6.0)             # back to the default tolerances
    assert min(emu.last_plan(len(sj))) < 0 and relerr(W6, W4) < 1e-13
    W7 = emu.cwt(x2[:2999], 1.0, sj, 1, 4.0)             # other wavelet family, same scales
    W7r = orc.cwt(x2[:2999], 1.0, wavelet=orc.Paul(4), freqs=1 / (orc.Paul(4).flambda() * sj[:20]))[0]
    assert W7r.shape[0] == 20 and relerr(W7[:20], W7r) < 1e-10   # (the largest scales are NaN rows for Paul)


def test_wide_band_expansion_plans(emu):
    """Coarse grids below 2x oversampling (band half-width up to 11/32 of Nc, 16-20 taps) are planned
    for fp64; a response that peaks off-centre in such a band (Paul) keeps the 2x rule (engine.cu:
    expand_gain).  Either way the coefficients match the oracle."""
    n = 2 ** 13
    rs = np.random.RandomState(21)
    x = rs.randn(n).cumsum() + 50.0          # red spectrum with a large mean: the hard case for the coarse grid
    # Morlet: band half-width hw = 8.58 / s * n / (2 pi) bins; Nc = n/8 = 1024: xi = hw / Nc
    for xi_target, expect_log2Nc in ((0.20, 10), (0.30, 10), (0.33, 10), (0.36, None)):
        s = 8.58 * n / (2 * np.pi) / (xi_target * 1024)
        sj = np.array([s, 1.01 * s])
        W = emu.cwt(x, 1.0, sj, 0, 6.0)
        plan = emu.last_plan(2)
        # beyond 11/32 the next coarse grid would be n/4 (expansion by four is off): pruned transform
        assert (plan[0] == -expect_log2Nc) if expect_log2Nc else (plan[0] > 0), (xi_target, plan)
        Wr = orc.cwt(x, 1.0, wavelet=orc.Morlet(6), freqs=1 / (orc.Morlet(6).flambda() * sj))[0]
        assert relerr(W, Wr) < 1e-12, (xi_target, relerr(W, Wr))
    # Paul(4): one-sided band [0, f_c / s], response peak at f = 4 of f_c ~ 51: far from the band centre
    m = orc.Paul(4)
    for s in (60.0, 80.0, 100.0, 140.0):
        sj = np.array([s])
        W = emu.cwt(x, 1.0, sj, 1, 4.0)
        Wr = orc.cwt(x, 1.0, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
        assert relerr(W, Wr) < 1e-12, (s, emu.last_plan(1), relerr(W, Wr))
