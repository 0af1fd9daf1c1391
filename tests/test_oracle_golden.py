"""Pins the CPU oracle (oracle/cwt_oracle.py) against fixtures produced by the real
reference (tests/golden/make_golden.py).  CPU only."""
import numpy as np
import pytest

from conftest import load_golden, relerr, golden_cwt_kwargs
from oracle import cwt_oracle as orc

CWT_CASES = ["nino3_morlet_tutorial", "nino3_morlet_default", "nino3_paul_default",
             "nino3_dog_default", "nino3_dog6", "nino3_dog3_odd", "nino3_morlet_f0_8",
             "chirp4000_morlet", "chirp4000_paul", "chirp4000_dog", "chirp32k_morlet",
             "chirp8k_f32_paul"]
TOL = 1e-12  # oracle vs reference: same algorithm, same FFT library


def mother_of(g):
    cls = {"morlet": orc.Morlet, "paul": orc.Paul, "dog": orc.DOG}[str(g["wavelet"])]
    return cls(int(g["param"]))


@pytest.mark.parametrize("name", CWT_CASES)
def test_cwt_matches_reference(name):
    g = load_golden(name)
    mother = mother_of(g)
    kw = golden_cwt_kwargs(g)
    W, sj, freqs, coi, fft, fftfreqs = orc.cwt(g["x"], float(g["dt"]), wavelet=mother, **kw)
    assert tuple(W.shape) == tuple(g["shape"])
    st = int(g["stride"])
    tol = 2e-6 if g["x"].dtype == np.float32 else TOL  # ref does the 1st FFT in c64
    assert relerr(W[:, ::st], g["W"]) < tol
    assert abs((np.abs(W) ** 2).sum() / float(g["power_sum"]) - 1) < max(tol, 1e-12) * 10
    np.testing.assert_array_equal(sj, g["sj"])
    np.testing.assert_array_equal(freqs, g["freqs"])
    np.testing.assert_allclose(coi, g["coi"], rtol=1e-15)
    assert relerr(fft, g["fft"]) < tol
    np.testing.assert_allclose(fftfreqs, g["fftfreqs"], rtol=1e-15)
    if "iW" in g.files:
        iW = orc.icwt(W, sj, float(g["dt"]), kw.get("dj", 1 / 12), mother)
        ist = int(g["iW_stride"]) if "iW_stride" in g.files else 1
        assert relerr(iW[::ist], g["iW"]) < max(tol, 1e-12)
        if ist > 1:
            assert abs((np.abs(iW) ** 2).sum() / float(g["iW_power_sum"]) - 1) < max(tol, 1e-12) * 10


NOPAD_CASES = ["nopad_nino3_morlet", "nopad_nino3_paul", "nopad_nino501_paul", "nopad_nino3_dog3",
               "nopad_chirp4001_morlet", "nopad_chirp3000_dog"]


@pytest.fixture
def unpadded_oracle(monkeypatch):
    """The oracle with the transform-length policy of the reference's pyfftw branch."""
    monkeypatch.setattr(orc, "PAD_NEXT_POW2", False)


@pytest.mark.parametrize("name", NOPAD_CASES)
def test_unpadded_cwt_matches_reference(unpadded_oracle, name):
    """Fixtures: the reference's own cwt/icwt run with `fft_kwargs -> {'n': len(signal)}`
    (helpers.py:15-19), see make_golden.py."""
    g = load_golden(name)
    mother = mother_of(g)
    kw = golden_cwt_kwargs(g)
    W, sj, freqs, coi, fft, fftfreqs = orc.cwt(g["x"], float(g["dt"]), wavelet=mother, **kw)
    assert tuple(W.shape) == tuple(g["shape"])
    st = int(g["stride"])
    assert relerr(W[:, ::st], g["W"]) < TOL
    np.testing.assert_array_equal(sj, g["sj"])
    assert fft.size == g["x"].size // 2 - 1 and relerr(fft, g["fft"]) < TOL
    np.testing.assert_allclose(fftfreqs, g["fftfreqs"], rtol=1e-15)
    if "iW" in g.files:
        assert relerr(orc.icwt(W, sj, float(g["dt"]), kw.get("dj", 1 / 12), mother), g["iW"]) < 1e-12


def test_unpadded_differs_from_padded_and_xwt(unpadded_oracle, monkeypatch):
    g = load_golden("nopad_ao_baltic_xwt")
    W12 = orc.xwt(g["y1"], g["y2"], float(g["dt"]), dj=1 / 12, wavelet=orc.Morlet(6))[0]
    assert relerr(W12, g["W12"]) < TOL
    monkeypatch.setattr(orc, "PAD_NEXT_POW2", True)
    W12p = orc.xwt(g["y1"], g["y2"], float(g["dt"]), dj=1 / 12, wavelet=orc.Morlet(6))[0]
    assert relerr(W12p, g["W12"]) > 1e-3     # the two policies really give different edges


def test_unpadded_coherence_and_smoothing(unpadded_oracle):
    g = load_golden("nopad_wct_smooth")
    m = orc.Morlet(6)
    assert relerr(m.smooth(g["Wr"], 1.0, 0.25, g["sj"]), g["Sr"]) < TOL
    assert relerr(m.smooth(g["Wc"], 1.0, 0.25, g["sj"]), g["Sc"]) < TOL
    WCT, aWCT, _, _, _ = orc.wct(g["y1"], g["y2"], float(g["dt"]), dj=1 / 12, sig=False, wavelet=m)
    assert relerr(WCT, g["WCT"]) < 1e-11 and relerr(aWCT, g["aWCT"]) < 1e-11
    sig95 = orc.wct_significance(0.2, 0.1, 1.0, 0.5, 2.0, 10, 0.95, m, mc_count=5,
                                 rng=np.random.RandomState(4321))
    np.testing.assert_allclose(sig95, g["sig95"], rtol=1e-12, equal_nan=True)


def test_known_anchors():
    """SURVEY 8c anchors measured on the reference."""
    g = load_golden("nino3_morlet_tutorial")
    assert tuple(g["shape"]) == (29, 504)
    assert abs(g["W"][0, 0] - (0.0324893658530221 + 0.13535815903662937j)) < 1e-15
    assert abs(float(g["power_sum"]) - 17916.846400687973) < 1e-8
    assert tuple(load_golden("nino3_paul_default")["shape"]) == (30, 504)
    assert tuple(load_golden("nino3_dog_default")["shape"]) == (41, 504)
    assert tuple(load_golden("nino3_morlet_default")["shape"]) == (33, 504)


def test_custom_freqs():
    g = load_golden("nino3_custom_freqs")
    W, sj, freqs, coi, _, _ = orc.cwt(g["x"], float(g["dt"]), wavelet=orc.Morlet(6),
                                      freqs=g["freqs_in"])
    assert relerr(W, g["W"]) < TOL
    np.testing.assert_array_equal(sj, g["sj"])


def test_xwt_wct():
    g = load_golden("ao_baltic_xwt_wct")
    y1, y2, dt = g["y1"], g["y2"], float(g["dt"])
    m = orc.Morlet(6)
    W12, coi, freq, signif = orc.xwt(y1, y2, dt, dj=1 / 12, significance_level=0.8646,
                                     wavelet=m)
    assert tuple(W12.shape) == (76, 147)
    assert relerr(W12, g["W12"]) < TOL
    np.testing.assert_allclose(signif, g["signif"], rtol=1e-12)
    np.testing.assert_allclose(coi, g["coi"], rtol=1e-14)
    W12n, _, _, sn = orc.xwt(y1, y2, dt, dj=1 / 12, wavelet=m, normalize=False)
    assert relerr(W12n, g["W12_nonorm"]) < TOL
    np.testing.assert_allclose(sn, g["signif_nonorm"], rtol=1e-12)
    WCT, aWCT, _, _, sig = orc.wct(y1, y2, dt, dj=1 / 12, sig=False, wavelet=m)
    assert relerr(WCT, g["WCT"]) < 1e-10
    assert relerr(aWCT, g["aWCT"]) < 1e-10
    assert sig.shape == (1,) and sig[0] == 0
    assert abs(orc.ar1(y1)[0] - float(g["a1"])) < 1e-14
    assert abs(float(g["a_nino"]) - 0.772491118627944) < 1e-12


def test_smooth():
    g = load_golden("smooth_cases")
    sj = g["sj"]
    Sr = orc.smooth(g["Wr"], 1.0, 0.25, sj)
    Sc = orc.smooth(g["Wc"], 1.0, 0.25, sj)
    assert Sr.dtype == np.float64 and np.iscomplexobj(Sc)
    assert relerr(Sr, g["Sr"]) < TOL
    assert relerr(Sc, g["Sc"]) < TOL


def test_wct_significance_seeded():
    g = load_golden("wct_significance_seed1234")
    np.random.seed(int(g["seed"]))
    sig = orc.wct_significance(float(g["al1"]), float(g["al2"]), dt=float(g["dt"]),
                               dj=float(g["dj"]), s0=float(g["s0"]), J=int(g["J"]),
                               significance_level=float(g["level"]),
                               mc_count=int(g["mc_count"]))
    assert relerr(sig, g["sig95"]) < 1e-12


def test_wct_sig_end_to_end_seeded():
    g = load_golden("wct_sig_seed99")
    np.random.seed(99)
    WCT, aWCT, coi, freq, sig = orc.wct(g["y1"], g["y2"], 1.0, dj=0.5, s0=2.0, J=8,
                                        sig=True, wavelet=orc.Morlet(6), mc_count=4)
    assert relerr(WCT, g["WCT"]) < 1e-10
    assert relerr(sig, g["sig"]) < 1e-12
