"""GPU parity tests of the cwt hot path: CUDA engine (through the C ABI / ctypes and the
pycwt-compatible Python surface) versus the golden fixtures produced by the real
reference and versus the CPU oracle on seeded inputs.

Tolerances (BASELINE.json north_star): fp64 engine 1e-10 relative to max|W_ref| (achieved
~1e-15); fp32 engine 1e-5 (achieved ~3e-7)."""
import numpy as np
import pytest

from conftest import load_golden, relerr, golden_cwt_kwargs
from _rowerr import check_rows
from oracle import cwt_oracle as orc

pytestmark = pytest.mark.gpu

TOL64 = 1e-10
TOL32 = 1e-5

CWT_CASES = ["nino3_morlet_tutorial", "nino3_morlet_default", "nino3_paul_default",
             "nino3_dog_default", "nino3_dog6", "nino3_dog3_odd", "nino3_morlet_f0_8",
             "chirp4000_morlet", "chirp4000_paul", "chirp4000_dog", "chirp32k_morlet",
             "chirp8k_f32_paul"]


@pytest.fixture(scope="module")
def pycwt():
    import pycwt_b200
    return pycwt_b200


def chirp(n):
    t = np.arange(n) / n
    return np.sin(2 * np.pi * (50 * t + (n / 8) * t ** 2))


def mothers(pycwt, g):
    name, p = str(g["wavelet"]), int(g["param"])
    return {"morlet": pycwt.Morlet, "paul": pycwt.Paul, "dog": pycwt.DOG}[name](p)


@pytest.mark.parametrize("name", CWT_CASES)
def test_cwt_golden(pycwt, name):
    g = load_golden(name)
    kw = golden_cwt_kwargs(g)
    W, sj, freqs, coi, fft, fftfreqs = pycwt.cwt(g["x"], float(g["dt"]),
                                                 wavelet=mothers(pycwt, g), **kw)
    assert W.dtype == np.complex128 and tuple(W.shape) == tuple(g["shape"])
    f32 = g["x"].dtype == np.float32  # the reference runs its first FFT in complex64
    tol = 2e-6 if f32 else TOL64
    st = int(g["stride"])
    assert relerr(W[:, ::st], g["W"]) < tol
    assert relerr(np.abs(W[:, ::st]) ** 2, np.abs(g["W"]) ** 2) < tol
    assert abs((np.abs(W) ** 2).sum() / float(g["power_sum"]) - 1) < 10 * tol
    np.testing.assert_array_equal(sj, g["sj"])
    np.testing.assert_array_equal(freqs, g["freqs"])
    np.testing.assert_array_equal(coi, g["coi"])
    assert relerr(fft, g["fft"]) < tol
    np.testing.assert_array_equal(fftfreqs, g["fftfreqs"])


def test_cwt_list_input_and_string_wavelet(pycwt):
    g = load_golden("nino3_morlet_default")
    W, sj, *_ = pycwt.cwt(list(g["x"]), 0.25, dj=0.25, wavelet="morlet")
    assert relerr(W, g["W"]) < TOL64
    with pytest.raises(KeyError):
        pycwt.cwt(g["x"], 0.25, wavelet="nosuchwavelet")


def test_custom_freqs(pycwt):
    g = load_golden("nino3_custom_freqs")
    W, sj, freqs, coi, _, _ = pycwt.cwt(g["x"], float(g["dt"]), wavelet=pycwt.Morlet(6),
                                        freqs=g["freqs_in"])
    assert relerr(W, g["W"]) < TOL64
    np.testing.assert_array_equal(sj, g["sj"])


def test_duck_typed_wavelet_uses_table_path(pycwt):
    """Any object with psi_ft/flambda/coi works (reference wavelet.py:650-663)."""
    class MyMorlet(object):  # not a subclass: no analytic engine path
        name = "mine"
        def psi_ft(self, f):
            return np.pi ** -0.25 * np.exp(-0.5 * (f - 5.0) ** 2)
        def flambda(self):
            return 4 * np.pi / (5.0 + np.sqrt(27.0))
        def coi(self):
            return 1 / np.sqrt(2)
    x = chirp(700) + 0.3 * np.random.RandomState(5).randn(700)
    W, sj, *_ = pycwt.cwt(x, 1.0, dj=0.25, wavelet=MyMorlet())
    Wr, sjr, *_ = orc.cwt(x, 1.0, dj=0.25, wavelet=orc.Morlet(5.0))
    np.testing.assert_allclose(sj, sjr, rtol=1e-15)
    assert relerr(W, Wr) < TOL64
    # long signal through the dense two-kernel path
    x = chirp(5000)
    W, sj, *_ = pycwt.cwt(x, 1.0, dj=0.5, wavelet=MyMorlet())
    Wr = orc.cwt(x, 1.0, dj=0.5, wavelet=orc.Morlet(5.0))[0]
    assert relerr(W, Wr) < TOL64


@pytest.mark.parametrize("n0", [2, 3, 5, 17, 31, 32, 33, 64, 100, 511, 1024, 1025, 2048,
                                4099, 10000, 2 ** 16])
def test_lengths_edge_cases(pycwt, n0):
    rs = np.random.RandomState(n0)
    x = rs.randn(n0)
    if n0 < 4:
        sj = np.array([1.0, 2.0, 3.5])
        eng = pycwt.default_engine()
        W = eng.cwt(x, 1.0, sj, 0, 6.0)
        npad = orc.next_pow2(n0)
        om = 2 * np.pi * np.fft.fftfreq(npad, 1.0)
        with np.errstate(all="ignore"):  # Np == 2: the reference's norm is NaN
            filt = (sj[:, None] * om[1] * npad) ** .5 * orc.Morlet(6).psi_ft(sj[:, None] * om)
            Wr = np.fft.ifft(np.fft.fft(x, npad) * filt, axis=1)[:, :n0]
        assert relerr(W, Wr) < TOL64
        return
    for mother, ref in ((pycwt.Morlet(6), orc.Morlet(6)), (pycwt.DOG(2), orc.DOG(2)),
                        (pycwt.Paul(4), orc.Paul(4))):
        W, sj, *_ = pycwt.cwt(x, 1.0, dj=0.5, wavelet=mother)
        with np.errstate(all="ignore"):
            Wr, sjr, *_ = orc.cwt(x, 1.0, dj=0.5, wavelet=ref)
        np.testing.assert_array_equal(sj, sjr)
        assert relerr(W, Wr) < TOL64


def test_all_plan_classes_exercised(pycwt):
    """One transform that uses every pruned length 2^5..2^16 and the dense path (exact mode:
    expansion path off), then the same transform in the default mode (expansion path on)."""
    from test_emu_exact import GATE
    noise = np.random.RandomState(1).randn(2 ** 16)
    x = chirp(2 ** 16) + 0.1 * noise
    Wr = orc.cwt(x, 1.0, dj=0.5, s0=2.0, J=30, wavelet=orc.Morlet(6))[0]
    eng = pycwt.default_engine()
    eng.set_expand_eps(0.0, 0.0)
    try:
        # every exact row on its own, on the chirp and on white noise alone
        for xx, ref in ((x, Wr), (noise, None)):
            W, sj, *_ = pycwt.cwt(xx, 1.0, dj=0.5, s0=2.0, J=30, wavelet=pycwt.Morlet(6))
            plan = eng.last_plan(len(sj))
            assert set(plan) >= set(range(5, 17)), plan
            if ref is None:
                ref = orc.cwt(xx, 1.0, dj=0.5, s0=2.0, J=30, wavelet=orc.Morlet(6))[0]
            err = check_rows(W, ref, *GATE[0], what="exact rows")
            print("exact rows: worst row error %.2e" % err)
    finally:
        eng.set_expand_eps()
    W, sj, *_ = pycwt.cwt(x, 1.0, dj=0.5, s0=2.0, J=30, wavelet=pycwt.Morlet(6))
    plan = eng.last_plan(len(sj))
    assert set(plan) >= set(range(-13, -5)) and max(plan) == 16, plan   # coarse grids 2^6..2^13
    assert relerr(W, Wr) < 2e-13
    # every expansion row on its own (the global maximum hides the small rows)
    rows = [i for i, p in enumerate(plan) if p < 0]
    err = check_rows(W[rows], Wr[rows], 1e-12, 1e-14, what="expansion rows")
    print("expansion rows: worst row error %.2e" % err)


def test_expansion_path_families_and_precisions(pycwt, monkeypatch):
    """Expansion rows of every family against the oracle, fp64 (alias bound 5e-13) and fp32."""
    x = chirp(2 ** 15) + 0.1 * np.random.RandomState(3).randn(2 ** 15)
    eng = pycwt.default_engine()
    cases = ((pycwt.Morlet(6), orc.Morlet(6), dict(s0=2.0, dj=0.5, J=26)),
             (pycwt.Paul(4), orc.Paul(4), dict(s0=2.0, dj=0.5, J=13)),
             (pycwt.DOG(2), orc.DOG(2), dict(s0=2.0, dj=0.5, J=26)),
             (pycwt.DOG(3), orc.DOG(3), dict(s0=2.0, dj=0.5, J=26)))
    for mother, ref, kw in cases:
        Wr = orc.cwt(x, 1.0, wavelet=ref, **kw)[0]
        W, sj, *_ = pycwt.cwt(x, 1.0, wavelet=mother, **kw)
        assert min(eng.last_plan(len(sj))) < 0
        assert relerr(W, Wr) < 2e-13, (type(mother).__name__, relerr(W, Wr))
    monkeypatch.setenv("CWTB_PRECISION", "fp32")
    for mother, ref, kw in cases:
        Wr = orc.cwt(x, 1.0, wavelet=ref, **kw)[0]
        W, sj, *_ = pycwt.cwt(x.astype(np.float32), 1.0, wavelet=mother, **kw)
        assert min(eng.last_plan(len(sj))) < 0
        assert relerr(W, Wr) < TOL32


def test_fp32_engine(pycwt, monkeypatch):
    """Config 3 flavour (SURVEY 8d): float32 chirp, Paul(4) and DOG(2), fp32 arithmetic."""
    monkeypatch.setenv("CWTB_PRECISION", "fp32")
    x = chirp(2 ** 14).astype(np.float32)
    for mother, ref, kw in ((pycwt.Paul(4), orc.Paul(4), dict(s0=1.4324, dj=1 / 6, J=40)),
                            (pycwt.DOG(2), orc.DOG(2), dict(s0=0.5033, dj=1 / 4, J=50)),
                            (pycwt.Morlet(6), orc.Morlet(6), dict(s0=2.0, dj=1 / 4, J=40))):
        W, sj, *_ = pycwt.cwt(x, 1.0, wavelet=mother, **kw)
        Wr = orc.cwt(x.astype(np.float64), 1.0, wavelet=ref, **kw)[0]
        err = relerr(W, Wr)
        assert err < TOL32, (type(mother).__name__, err)


def test_band_eps_exact_mode_matches(pycwt):
    """eps = 0 keeps every representable bin; results agree with the default pruning to
    far below the parity tolerance."""
    x = chirp(4096) + 0.2 * np.random.RandomState(2).randn(4096)
    eng = pycwt.default_engine()
    sj = 2.0 * 2 ** (np.arange(40) / 4.0)
    W0 = eng.cwt(x, 1.0, sj, 0, 6.0)
    eng.set_band_eps(0.0)
    try:
        W1 = eng.cwt(x, 1.0, sj, 0, 6.0)
    finally:
        eng.set_band_eps(1e-16)
    assert relerr(W0, W1) < 1e-14
    Wr = orc.cwt(x, 1.0, dj=0.25, s0=2.0, J=39, wavelet=orc.Morlet(6))[0]
    assert relerr(W1, Wr) < TOL64


def test_nan_signal_propagates(pycwt):
    x = np.random.RandomState(0).randn(300)
    x[17] = np.nan
    W, sj, *_ = pycwt.cwt(x, 1.0, dj=0.5)
    assert np.isnan(W).all() and W.shape[0] == len(sj)


def test_linearity_and_parseval_full_size(pycwt):
    """Size-independent properties at the north-star size (N = 2^20, fp64, Morlet):
    linearity of the transform and Parseval per scale
        sum_n |W_j[n]|^2 = (1/Np) sum_k |x^_k|^2 |psi^_j,k|^2   (n0 = Np here),
    checked with numpy on the host for a handful of rows fetched from the device."""
    n = 2 ** 20
    eng = pycwt.default_engine()
    rs = np.random.RandomState(11)
    a = chirp(n)
    b = rs.randn(n)
    sj = 2.0 * 2 ** (np.arange(0, 256, 17) / 16.0)  # 16 scales spanning all classes
    Wa = eng.cwt(a, 1.0, sj, 0, 6.0)
    Wb = eng.cwt(b, 1.0, sj, 0, 6.0)
    Wab = eng.cwt(2.0 * a - 0.5 * b, 1.0, sj, 0, 6.0)
    assert relerr(Wab, 2.0 * Wa - 0.5 * Wb) < 1e-12
    om = 2 * np.pi * np.fft.fftfreq(n, 1.0)
    xh = np.fft.fft(b)
    for j, s in enumerate(sj):
        filt = np.sqrt(s * om[1] * n) * orc.Morlet(6).psi_ft(s * om)
        rhs = (np.abs(xh * filt) ** 2).sum() / n
        lhs = (np.abs(Wb[j]) ** 2).sum()
        assert abs(lhs / rhs - 1) < 1e-11, (j, s, lhs, rhs)
    # spot parity against the oracle on 3 rows (full-length CPU inverse FFTs)
    rows = [0, 7, 15]
    filt = np.sqrt(sj[rows, None] * om[1] * n) * orc.Morlet(6).psi_ft(sj[rows, None] * om)
    Wr = np.fft.ifft(xh * filt, axis=1)
    assert relerr(Wb[rows], Wr) < TOL64


def test_signal_longer_than_2_20(pycwt):
    """n0 > 2^20 (Np = 2^21, 2^22): three-level path for the forward FFT and the dense scales."""
    rs = np.random.RandomState(8)
    for n0 in (2 ** 20 + 4321, 2 ** 22):
        x = chirp(n0) + 0.2 * rs.randn(n0)
        sj = np.array([2.0, 4.5, 20.0, 900.0, 3e4, 4e5])
        eng = pycwt.default_engine()
        W = eng.cwt(x, 1.0, sj, 0, 6.0)
        m = orc.Morlet(6)
        Wr = orc.cwt(x, 1.0, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
        assert relerr(W, Wr) < TOL64
    W, sj, freqs, coi, fft, fftfreqs = pycwt.cwt(x[:2 ** 20 + 9], 1.0, dj=2.0, wavelet="dog")
    Wr, sjr, _, _, fftr, _ = orc.cwt(x[:2 ** 20 + 9], 1.0, dj=2.0, wavelet=orc.DOG(2))
    assert relerr(W, Wr) < TOL64 and relerr(fft, fftr) < 1e-12


def test_engine_c2c_hook(pycwt):
    eng = pycwt.default_engine()
    rs = np.random.RandomState(4)
    for n in (2, 8, 64, 512, 1024, 4096, 2 ** 15, 2 ** 20, 2 ** 22):
        x = rs.randn(2, n) + 1j * rs.randn(2, n)
        assert relerr(eng.fft_c2c(x, -1), np.fft.fft(x, axis=1)) < 1e-13
        assert relerr(eng.fft_c2c(x, +1), np.fft.ifft(x, axis=1) * n) < 1e-13
        assert relerr(eng.fft_c2c(x, -1, precision=1), np.fft.fft(x, axis=1)) < 5e-6


def test_resident_transform_products(pycwt):
    """SURVEY 8f rank 2: power, rectified power, global spectrum (also inside the COI),
    scale-averaged power and icwt evaluated on the device-resident transform equal the NumPy
    arithmetic of pycwt/sample/simple_sample.py:64-91 on the oracle's W."""
    from test_emu_kernels import check_resident_products
    check_resident_products(pycwt.default_engine(), TOL64)


def test_resident_products_full_size(pycwt):
    """North-star size: the reductions agree with NumPy on rows fetched from the device,
    and the fp32 transform comes back as complex128 through the widening fetch."""
    n = 2 ** 20
    x = chirp(n)
    r = pycwt.cwt_resident(x, 1.0, 1 / 16, 2.0, 255, pycwt.Morlet(6))
    glbl = r.global_power()
    savg = r.scale_avg_power(16.0, 64.0, variance=1.0)
    inside = r.global_power(inside_coi=True)
    eng = r.engine
    rows = [0, 100, 255]
    per = r.period
    lo, hi = r.coi_ranges()
    for j in rows:
        Wj = np.empty((1, n), dtype=np.complex128)
        eng._check(eng.lib.cwtb_get_w(eng.h, Wj.ctypes.data, 1, j, 1))
        p = np.abs(Wj[0]) ** 2
        assert abs(glbl[j] / p.mean() - 1) < 1e-12
        assert np.array_equal(np.nonzero(per[j] <= r.coi)[0][[0, -1]], [lo[j], hi[j] - 1])
        assert abs(inside[j] / p[lo[j]:hi[j]].mean() - 1) < 1e-12
    sel = np.nonzero((per >= 16.0) & (per < 64.0))[0]
    acc = np.zeros(n)
    for j in sel:
        Wj = np.empty((1, n), dtype=np.complex128)
        eng._check(eng.lib.cwtb_get_w(eng.h, Wj.ctypes.data, 1, int(j), 1))
        acc += np.abs(Wj[0]) ** 2 / r.scales[j]
    acc *= r.dj * r.dt / r.wavelet.cdelta
    assert relerr(savg, acc) < 1e-12


def test_fp32_fetch_widening_large(pycwt, monkeypatch):
    """fp32 engine, complex128 result larger than one staging chunk (two-stream widening)."""
    monkeypatch.setenv("CWTB_PRECISION", "fp32")
    x = chirp(2 ** 18).astype(np.float32)
    kw = dict(s0=0.5033, dj=1 / 8, J=127)
    W, sj, *_ = pycwt.cwt(x, 1.0, wavelet=pycwt.DOG(2), **kw)
    assert W.dtype == np.complex128 and W.shape == (128, 2 ** 18)
    eng = pycwt.default_engine()
    W32 = eng.get_w(128, 2 ** 18, precision=1, out_f64=False)
    assert W32.dtype == np.complex64
    assert np.array_equal(W, W32.astype(np.complex128))
    rows = [0, 64, 127]
    om = 2 * np.pi * np.fft.fftfreq(2 ** 18, 1.0)
    xh = np.fft.fft(x.astype(np.float64))
    filt = np.sqrt(sj[rows, None] * om[1] * 2 ** 18) * np.conj(orc.DOG(2).psi_ft(sj[rows, None] * om))
    assert relerr(W[rows], np.fft.ifft(xh * filt, axis=1)) < TOL32


def test_unpadded_mode(pycwt):
    """SURVEY 8f rank 3: transforms at the signal's own length (the reference's pyfftw policy,
    helpers.py:15-19) against fixtures produced by the reference's own code with that policy."""
    from test_emu_kernels import check_unpadded_mode
    check_unpadded_mode(pycwt.default_engine(), TOL64)


def test_unpadded_long_signal_and_any_length_dft(pycwt):
    """Un-padded transform whose convolution length needs the two-kernel FFT (L = 2^18), rows
    checked against direct numpy DFTs; and the DFT hook for awkward lengths."""
    from pycwt_b200 import helpers
    eng = pycwt.default_engine()
    rs = np.random.RandomState(2)
    for n in [3, 7, 1000, 4099, 65537, 100003]:
        x = rs.randn(2, n) + 1j * rs.randn(2, n)
        assert relerr(eng.fft_c2c(x, -1), np.fft.fft(x, axis=1)) < 1e-12, n
    n = 100000
    x = chirp(n) + 0.1 * rs.randn(n)
    helpers.set_fft_padding(False)
    try:
        W, sj, *_ = pycwt.cwt(x, 1.0, 0.5, 2.0, 24, pycwt.Morlet(6))
    finally:
        helpers.set_fft_padding(True)
    om = 2 * np.pi * np.fft.fftfreq(n, 1.0)
    xh = np.fft.fft(x)
    rows = [0, 11, 24]
    filt = np.sqrt(sj[rows, None] * om[1] * n) * orc.Morlet(6).psi_ft(sj[rows, None] * om)
    assert relerr(W[rows], np.fft.ifft(xh * filt, axis=1)) < TOL64
    Wp = pycwt.cwt(x, 1.0, 0.5, 2.0, 24, pycwt.Morlet(6))[0]
    assert relerr(Wp[rows], W[rows]) > 1e-6      # padded and un-padded differ at the edges


def test_overlapped_fetch_equals_plain_fetch(pycwt):
    """Engine.cwt(fetch=True) copies the rows of the single-kernel chain back while the two-kernel
    chains still run; the result must be bit-identical to transform-then-fetch."""
    eng = pycwt.default_engine()
    n = 2 ** 17
    x = chirp(n) + 0.05 * np.random.RandomState(8).randn(n)
    sj = 2.0 * 2 ** (np.arange(0, 120) / 8.0)          # every class, ascending scales
    W1 = eng.cwt(x, 1.0, sj, 0, 6.0)
    eng.cwt(x, 1.0, sj, 0, 6.0, fetch=False)
    W2 = eng.get_w(sj.size, n)
    assert np.array_equal(W1, W2)
    perm = np.random.RandomState(9).permutation(sj.size)  # unordered scales: plain sequence
    W3 = eng.cwt(x, 1.0, sj[perm], 0, 6.0)
    assert np.array_equal(W3, W1[perm])
    assert eng.last_kernel_ms() > 0


def test_expansion_by_four(monkeypatch):
    """R = Np/Nc = 4 is off by default (no gain); both expansion kernels implement it
    (CWTB_EXPAND_MIN_R=2): the tensor-core kernel's 2-positions-by-4-phases column layout and the
    scalar kernel must give the same coefficients as the oracle."""
    from pycwt_b200 import _engine
    n = 2 ** 14
    x = chirp(n) + 0.1 * np.random.RandomState(4).randn(n)
    sj = 2.0 * 2 ** (np.arange(8, 40) / 4.0)
    Wr = orc.cwt(x, 1.0, wavelet=orc.Morlet(6), freqs=1 / (orc.Morlet(6).flambda() * sj))[0]
    monkeypatch.setenv("CWTB_EXPAND_MIN_R", "2")
    for mma in ("1", "0"):
        monkeypatch.setenv("CWTB_EXPAND_MMA", mma)
        eng = _engine.Engine(0)
        try:
            W = eng.cwt(x, 1.0, sj, _engine.MORLET, 6.0)
            plan = eng.last_plan(len(sj))
            assert -12 in plan, plan          # coarse grids of Np/4 points are in play
            assert relerr(W, Wr) < TOL64, (mma, relerr(W, Wr))
        finally:
            eng.close()
