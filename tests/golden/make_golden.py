#!/usr/bin/env python
"""Generate golden fixtures from the REAL reference (regeirk/pycwt).

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

It imports the unmodified reference package from /root/reference, runs it on
fixed inputs and writes small `.npz` fixtures next to this file.  The reference
cannot travel to the GPU box, the fixtures can.  Inputs that come from the
reference's sample data files (NINO3 SST, AO, Baltic ice) are stored inside the
fixtures as plain arrays so that tests never read /root/reference.

Large outputs are stored column-subsampled (`W[:, ::stride]`) together with the
full-array power sum, to keep the committed blobs small; where that still leaves a fixture
above 1 MB, the inverse transform is stored as `iW[::iW_stride]` with its power sum too.
"""
import os
import sys
import warnings

import numpy as np

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")
import pycwt  # noqa: E402  (the reference)
from pycwt.helpers import ar1  # noqa: E402


def chirp(n):
    t = np.arange(n) / n
    return np.sin(2 * np.pi * (50 * t + (n / 8) * t ** 2))


def save(name, **arrays):
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **arrays)
    print("%-28s %8.1f KB" % (name, os.path.getsize(path) / 1024))


def cwt_case(name, x, dt, wavelet_name, param, stride=1, iw_stride=1, **kw):
    cls = {"morlet": pycwt.Morlet, "paul": pycwt.Paul, "dog": pycwt.DOG}[wavelet_name]
    mother = cls(param)
    W, sj, freqs, coi, fft, fftfreqs = pycwt.cwt(x, dt, wavelet=mother, **kw)
    extra = {}
    if wavelet_name != "paul" or param == 4:
        if mother.cdelta != -1:
            iW = pycwt.icwt(W, sj, dt, kw.get("dj", 1 / 12), mother)
            extra["iW"] = iW[::iw_stride]
            if iw_stride > 1:
                extra.update(iW_stride=iw_stride, iW_power_sum=(np.abs(iW) ** 2).sum())
    save(name, x=np.asarray(x), dt=dt, wavelet=wavelet_name, param=param,
         kw_keys=np.array(sorted(kw.keys())),
         kw_vals=np.array([kw[k] for k in sorted(kw.keys())], dtype=float),
         W=W[:, ::stride], stride=stride, power_sum=(np.abs(W) ** 2).sum(),
         shape=np.array(W.shape), sj=sj, freqs=freqs, coi=coi, fft=fft,
         fftfreqs=fftfreqs, **extra)


def main():
    nino = np.loadtxt(os.path.join(REF, "pycwt/sample/sst_nino3.dat"))
    # config 1 (SURVEY 8d): tutorial call and defaults for the three families
    cwt_case("nino3_morlet_tutorial", nino, 0.25, "morlet", 6, dj=0.25, s0=0.5, J=28)
    cwt_case("nino3_morlet_default", nino, 0.25, "morlet", 6, dj=0.25)
    cwt_case("nino3_paul_default", nino, 0.25, "paul", 4, dj=0.25)   # drops NaN rows
    cwt_case("nino3_dog_default", nino, 0.25, "dog", 2, dj=0.25)
    cwt_case("nino3_dog6", nino, 0.25, "dog", 6, dj=0.25)
    cwt_case("nino3_dog3_odd", nino, 0.25, "dog", 3, dj=0.5)          # imaginary psi_ft
    cwt_case("nino3_morlet_f0_8", nino, 0.25, "morlet", 8, dj=0.5)
    # non power-of-two length, multi-kernel sizes, sub-sampled output
    x = chirp(4000) + 0.1 * np.random.RandomState(3).randn(4000)
    cwt_case("chirp4000_morlet", x, 1.0, "morlet", 6, stride=8, dj=1 / 8, s0=2.0, J=72)
    cwt_case("chirp4000_paul", x, 1.0, "paul", 4, stride=8, dj=1 / 8)  # NaN rows dropped
    cwt_case("chirp4000_dog", x, 1.0, "dog", 2, stride=8, dj=1 / 8, s0=0.5033, J=80)
    x = chirp(2 ** 15)
    cwt_case("chirp32k_morlet", x, 1.0, "morlet", 6, stride=128, iw_stride=8, dj=1 / 4, s0=2.0, J=52)
    x32 = chirp(2 ** 13).astype(np.float32)
    cwt_case("chirp8k_f32_paul", x32, 1.0, "paul", 4, stride=16, dj=1 / 6, s0=1.4324, J=40)
    # custom frequencies
    fr = np.linspace(0.4, 0.01, 17)
    mother = pycwt.Morlet(6)
    W, sj, freqs, coi, fft, fftfreqs = pycwt.cwt(nino, 0.25, wavelet=mother, freqs=fr)
    save("nino3_custom_freqs", x=nino, dt=0.25, freqs_in=fr, W=W, sj=sj, freqs=freqs,
         coi=coi)

    # significance() for the three test kinds + helper functions (host-side O(S) rows)
    mother = pycwt.Morlet(6)
    W, sj, freqs, coi, fft, fftfreqs = pycwt.cwt(nino, 0.25, 0.25, 0.5, 28, mother)
    std = nino.std()
    dat_norm = nino / std
    alpha = ar1(nino)[0]
    s0_, f0_ = pycwt.significance(1.0, 0.25, sj, 0, alpha, significance_level=0.95, wavelet=mother)
    s1_, f1_ = pycwt.significance(std ** 2, 0.25, sj, 1, alpha, significance_level=0.95,
                                  dof=nino.size - sj, wavelet=mother)
    s2_, f2_ = pycwt.significance(std ** 2, 0.25, sj, 2, alpha, significance_level=0.95,
                                  dof=[sj[3], sj[13]], wavelet=mother)
    s3_, f3_ = pycwt.significance(dat_norm, 0.25, sj, 0, significance_level=0.9, wavelet=mother)
    from pycwt.helpers import ar1_spectrum, rect
    save("significance_nino3", x=nino, sj=sj, alpha=alpha, ar1_full=np.array(ar1(nino)),
         s0=s0_, f0=f0_, s1=s1_, f1=f1_, s2=s2_, f2=f2_, s3=s3_, f3=f3_,
         spec=ar1_spectrum(freqs * 0.25, alpha), rect7=rect(7, normalize=True), rect2=rect(2))

    # xwt / wct on the AO x Baltic sample (sample_xwt.py preprocessing minus boxpdf,
    # which raises NameError in the reference)
    t1, s1 = np.loadtxt(os.path.join(REF, "pycwt/sample/jao.dat"), unpack=True)
    t2, s2 = np.loadtxt(os.path.join(REF, "pycwt/sample/jbaltic.dat"), unpack=True)
    dt = np.diff(t1)[0]
    n = min(t1.size, t2.size)
    s1, s2 = s1[:n], s2[:n]
    mother = pycwt.Morlet(6)
    W12, coi, freq, signif = pycwt.xwt(s1, s2, dt, dj=1 / 12, s0=-1, J=-1,
                                       significance_level=0.8646, wavelet=mother,
                                       normalize=True)
    WCT, aWCT, coi2, freq2, sig = pycwt.wct(s1, s2, dt, dj=1 / 12, s0=-1, J=-1,
                                            sig=False, wavelet=mother, normalize=True)
    W12n, _, _, signifn = pycwt.xwt(s1, s2, dt, dj=1 / 12, wavelet=mother,
                                    normalize=False)
    save("ao_baltic_xwt_wct", y1=s1, y2=s2, dt=dt, W12=W12, coi=coi, freq=freq,
         signif=signif, WCT=WCT, aWCT=aWCT, sig=sig, W12_nonorm=W12n,
         signif_nonorm=signifn, a1=ar1(s1)[0], a2=ar1(s2)[0], a_nino=ar1(nino)[0])

    # Morlet.smooth on its own (real and complex input), n not a power of two and
    # n a power of two (circular case)
    rs = np.random.RandomState(7)
    sj = 2.0 * 2 ** (np.arange(0, 25) / 4.0)
    Wr = rs.rand(25, 300)
    Wc = rs.randn(25, 256) + 1j * rs.randn(25, 256)
    save("smooth_cases", sj=sj, dt=1.0, dj=0.25, Wr=Wr, Wc=Wc,
         Sr=mother.smooth(Wr, 1.0, 0.25, sj), Sc=mother.smooth(Wc, 1.0, 0.25, sj))

    # wct_significance with numpy's global RNG seeded (white surrogates, see
    # SURVEY 8a row 10).  Small problem so the reference's Python histogram
    # loop finishes in seconds.
    np.random.seed(1234)
    sig95 = pycwt.wct_significance(0.2, 0.1, dt=1.0, dj=0.5, s0=2.0, J=10,
                                   significance_level=0.95, wavelet=mother,
                                   mc_count=6, progress=False, cache=False)
    save("wct_significance_seed1234", al1=0.2, al2=0.1, dt=1.0, dj=0.5, s0=2.0, J=10,
         level=0.95, mc_count=6, seed=1234, sig95=sig95)

    # wct end-to-end with sig=True through the same seeded RNG
    np.random.seed(99)
    ya = rs.randn(200).cumsum()
    yb = ya + rs.randn(200)
    WCT, aWCT, coi, freq, sig = pycwt.wct(ya, yb, 1.0, dj=0.5, s0=2.0, J=8, sig=True,
                                          wavelet=mother, mc_count=4, progress=False,
                                          cache=False)
    save("wct_sig_seed99", y1=ya, y2=yb, WCT=WCT, aWCT=aWCT, coi=coi, freq=freq, sig=sig)

    # Un-padded transforms: the reference's own cwt/icwt/xwt code with the transform-length
    # policy of its pyfftw branch (helpers.py:15-19: n = len(signal)).  pyfftw is not installed
    # here, so the policy function is swapped in while the FFT library stays scipy's -- both are
    # exact DFTs of the requested length.
    import pycwt.wavelet as ref_wavelet
    import pycwt.mothers as ref_mothers
    padded_policy = ref_wavelet.fft_kwargs
    unpadded = lambda signal, **kw: {"n": len(signal)}   # noqa: E731
    ref_wavelet.fft_kwargs = unpadded
    ref_mothers.fft_kwargs = unpadded
    try:
        cwt_case("nopad_nino3_morlet", nino, 0.25, "morlet", 6, dj=0.25, s0=0.5, J=28)
        cwt_case("nopad_nino3_paul", nino, 0.25, "paul", 4, dj=0.25)
        cwt_case("nopad_nino3_dog3", nino, 0.25, "dog", 3, dj=0.5)
        # odd length + Paul: the all-NaN rows come from the most negative bin, -(n-1)/2
        cwt_case("nopad_nino501_paul", nino[:501], 0.25, "paul", 4, dj=0.25)
        x = chirp(4001) + 0.1 * np.random.RandomState(3).randn(4001)      # odd length
        cwt_case("nopad_chirp4001_morlet", x, 1.0, "morlet", 6, stride=8, dj=1 / 8, s0=2.0, J=72)
        cwt_case("nopad_chirp3000_dog", x[:3000], 1.0, "dog", 2, stride=8, dj=1 / 4, s0=0.5033, J=40)
        W12, coi, freq, signif = pycwt.xwt(s1, s2, dt, dj=1 / 12, wavelet=pycwt.Morlet(6))
        save("nopad_ao_baltic_xwt", y1=s1, y2=s2, dt=dt, W12=W12, coi=coi, freq=freq, signif=signif)
        # coherence and smoothing: the Gaussian time filter is circular at the rows' own length
        WCT, aWCT, coi2, freq2, sig = pycwt.wct(s1, s2, dt, dj=1 / 12, s0=-1, J=-1, sig=False,
                                                wavelet=pycwt.Morlet(6), normalize=True)
        rs2 = np.random.RandomState(7)
        sjs = 2.0 * 2 ** (np.arange(0, 25) / 4.0)
        Wr = rs2.rand(25, 300)
        Wc = rs2.randn(25, 301) + 1j * rs2.randn(25, 301)
        mo = pycwt.Morlet(6)
        np.random.seed(4321)
        sig95 = pycwt.wct_significance(0.2, 0.1, dt=1.0, dj=0.5, s0=2.0, J=10,
                                       significance_level=0.95, wavelet=mo,
                                       mc_count=5, progress=False, cache=False)
        save("nopad_wct_smooth", y1=s1, y2=s2, dt=dt, WCT=WCT, aWCT=aWCT, sj=sjs, Wr=Wr, Wc=Wc,
             Sr=mo.smooth(Wr, 1.0, 0.25, sjs), Sc=mo.smooth(Wc, 1.0, 0.25, sjs), sig95=sig95)
    finally:
        ref_wavelet.fft_kwargs = padded_policy
        ref_mothers.fft_kwargs = padded_policy


if __name__ == "__main__":
    main()
