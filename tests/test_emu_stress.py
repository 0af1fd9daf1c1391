"""Randomised parity sweep of the kernel logic (CPU, host-emulation build, see
tests/test_emu_kernels.py for what that is): random lengths, sampling intervals, unordered
scale sets from sub-Nyquist to beyond the record length, all wavelet families and orders,
both engine precisions.  Reference = the numpy formula of pycwt/wavelet.py:102-106.

The loop bodies are check_* functions that take an engine: tests/test_gpu_expansion.py runs
them with the same seeds on the B200, where the planner differs (tensor-core expansion kernel,
tap counts rounded to its k-steps, 20-tap coarse grids).  Every row is gated on its own
(tests/_rowerr.py), the inputs are white noise."""
import numpy as np
import pytest

from conftest import ROOT
from _rowerr import check_rows
from oracle import cwt_oracle as orc

# row gates (tests/_rowerr.py): (tol_row, tol_abs) per engine precision
ROW_GATE = {0: (1e-10, 1e-13), 1: (3e-5, 3e-6)}


@pytest.fixture(scope="module")
def emu():
    import os
    from pycwt_b200 import build as _build, _engine
    eng = _engine.Engine(0, lib_path=_build.build_emulation(os.path.join(ROOT, "tests", "_emu")))
    yield eng
    eng.close()


def check_random_transforms(eng, seed, log2_max=15.5, draws=60):
    """Random padded transforms against the numpy formula; returns (checked, worst row error
    per precision)."""
    rs = np.random.RandomState(seed)
    checked = 0
    worst = {0: 0.0, 1: 0.0}
    for _ in range(draws):
        n0 = max(4, int(2 ** rs.uniform(2.1, log2_max)))
        dt = float(10 ** rs.uniform(-2, 2))
        fam = rs.randint(3)
        if fam == 0:
            par = float(rs.choice([6, 6, 4.5, 8, 12, 20, 1.5]))
            mo = orc.Morlet(par)
        elif fam == 1:
            par = int(rs.choice([4, 1, 2, 6, 10]))
            mo = orc.Paul(par)
        else:
            par = int(rs.choice([2, 1, 3, 6, 9]))
            mo = orc.DOG(par)
        S = rs.randint(1, 30)
        sj = dt * 2 ** rs.uniform(-1, np.log2(n0) + 3, size=S)
        x = rs.randn(n0) * 10 ** rs.uniform(-3, 3)
        prec = int(rs.rand() < 0.3)
        npad = orc.next_pow2(n0)
        om = 2 * np.pi * np.fft.fftfreq(npad, dt)
        with np.errstate(all="ignore"):
            filt = (sj[:, None] * om[1] * npad) ** .5 * np.conj(mo.psi_ft(sj[:, None] * om))
            Wr = np.fft.ifft(np.fft.fft(x, npad) * filt, axis=1)[:, :n0]
        ok = ~np.isnan(Wr).any(axis=1)     # rows the reference would drop (Paul overflow)
        # degenerate draws: every scale so far beyond the record that the whole transform is
        # below 1e-15 of the signal (under the band cut-off by design, and under the fp32 range)
        if not ok.any() or np.abs(Wr[ok]).max() < 1e-15 * np.abs(x).max():
            continue
        W = eng.cwt(x, dt, sj, fam, par, prec)
        err = check_rows(W[ok], Wr[ok], *ROW_GATE[prec], what=(n0, dt, fam, par, S, prec))
        worst[prec] = max(worst[prec], err)
        checked += 1
    return checked, worst


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_random_transforms(emu, seed):
    checked, worst = check_random_transforms(emu, seed)
    print("seed %d: worst row error fp64 %.2e, fp32 %.2e" % (seed, worst[0], worst[1]))
    assert checked > 40


def check_random_unpadded_transforms(eng, seed):
    """Same sweep for the un-padded policy (helpers.py:15-19): transform length = n0, any n0
    (odd, prime, smooth), through the Bluestein path; plus the any-length DFT hook."""
    rs = np.random.RandomState(seed)
    worst = 0.0
    eng.set_padding(False)
    try:
        checked = 0
        for _ in range(40):
            n0 = max(3, int(2 ** rs.uniform(1.6, 13.5)))
            dt = float(10 ** rs.uniform(-2, 2))
            fam = rs.randint(3)
            if fam == 0:
                par = float(rs.choice([6, 6, 4.5, 8, 12]))
                mo = orc.Morlet(par)
            elif fam == 1:
                par = int(rs.choice([4, 1, 2, 6]))
                mo = orc.Paul(par)
            else:
                par = int(rs.choice([2, 1, 3, 6]))
                mo = orc.DOG(par)
            S = rs.randint(1, 12)
            sj = dt * 2 ** rs.uniform(-1, np.log2(n0) + 2, size=S)
            x = rs.randn(n0) * 10 ** rs.uniform(-3, 3)
            om = 2 * np.pi * np.fft.fftfreq(n0, dt)
            with np.errstate(all="ignore"):
                filt = (sj[:, None] * om[1] * n0) ** .5 * np.conj(mo.psi_ft(sj[:, None] * om))
                Wr = np.fft.ifft(np.fft.fft(x) * filt, axis=1)
            ok = ~np.isnan(Wr).any(axis=1)
            if not ok.any() or np.abs(Wr[ok]).max() < 1e-15 * np.abs(x).max():
                continue
            W = eng.cwt(x, dt, sj, fam, par, 0)
            assert eng.padded_length() == (n0 if n0 & (n0 - 1) else n0)
            err = check_rows(W[ok], Wr[ok], *ROW_GATE[0], what=(n0, dt, fam, par, S))
            worst = max(worst, err)
            spec = eng.signal_fft()
            ref = np.fft.fft(x)[1:n0 // 2] / np.sqrt(n0)
            if ref.size:
                assert np.abs(spec - ref).max() <= 1e-12 * max(np.abs(ref).max(), 1e-300)
            checked += 1
        assert checked > 25
        for n in rs.randint(3, 3000, size=12):
            z = rs.randn(1, int(n)) + 1j * rs.randn(1, int(n))
            assert np.abs(eng.fft_c2c(z, -1) - np.fft.fft(z, axis=1)).max() < 1e-12 * n
    finally:
        eng.set_padding(True)
    return worst


@pytest.mark.parametrize("seed", [21, 22])
def test_random_unpadded_transforms(emu, seed):
    print("seed %d: worst row error %.2e" % (seed, check_random_unpadded_transforms(emu, seed)))


def check_random_pairs_smoothing_and_batches(eng, seed):
    """Randomised shapes through the cross-wavelet, coherence, smoothing and batched entry
    points (both transform-length policies), against the oracle."""
    rs = np.random.RandomState(seed)
    m = orc.Morlet(6)
    for it in range(14):
        pad = bool(rs.rand() < 0.6)
        eng.set_padding(pad)
        orc.PAD_NEXT_POW2 = pad
        try:
            n = int(2 ** rs.uniform(4.5, 12.5))
            dt = float(10 ** rs.uniform(-1, 1))
            dj = float(rs.choice([0.5, 0.25, 1 / 6]))
            s0 = 2 * dt
            J = int(rs.randint(4, int(np.log2(n) / dj)))
            sj = s0 * 2 ** (np.arange(J + 1) * dj)
            y1 = rs.randn(n).cumsum()
            y2 = np.roll(y1, 3) + rs.randn(n)
            klen = int(np.round(m.deltaj0 / dj * 2))
            # xwt: W1 conj(W2)
            W12 = eng.xwt(y1, y2, dt, sj, 0, 6.0)
            W1 = orc.cwt(y1, dt, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
            W2 = orc.cwt(y2, dt, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
            ref = W1 * W2.conj()
            check_rows(W12, ref, *ROW_GATE[0], what=("xwt", it, n, pad))
            # smoothing operator on its own (complex and real input)
            S = eng.smooth(ref, dt, sj, klen)
            Sr = m.smooth(ref, dt, dj, sj)
            assert np.abs(S - Sr).max() < 1e-10 * np.abs(Sr).max(), (it, n, pad)
            P = np.abs(W1) ** 2
            assert np.abs(eng.smooth(P, dt, sj, klen) - m.smooth(P, dt, dj, sj)).max() < 1e-10 * P.max()
            # coherence
            WCT, aWCT = eng.wct(y1, y2, dt, dj, sj, 0, 6.0, klen)
            inv = 1 / sj[:, None]
            R = np.abs(m.smooth(ref * inv, dt, dj, sj)) ** 2 / (
                m.smooth(np.abs(W1) ** 2 * inv, dt, dj, sj) * m.smooth(np.abs(W2) ** 2 * inv, dt, dj, sj))
            assert np.abs(WCT - R).max() < 1e-8, (it, n, pad, np.abs(WCT - R).max())
            assert np.abs(np.exp(1j * aWCT) - np.exp(1j * np.angle(ref))).max() < 1e-8
            # batched channels (padded policy only) equal per-channel transforms
            if pad and n >= 32:
                X = rs.randn(3, n)
                power, Wb = eng.cwt_batch(X, dt, sj, 0, 6.0, 0, want_power=True, want_w=True)
                for ch in range(3):
                    Wc = orc.cwt(X[ch], dt, wavelet=m, freqs=1 / (m.flambda() * sj))[0]
                    check_rows(Wb[ch], Wc, *ROW_GATE[0], what=("batch", it, n, ch))
                    assert np.allclose(power[ch], (np.abs(Wc) ** 2).mean(axis=1), rtol=1e-10)
        finally:
            eng.set_padding(True)
            orc.PAD_NEXT_POW2 = True


@pytest.mark.parametrize("seed", [31, 32])
def test_random_pairs_smoothing_and_batches(emu, seed):
    check_random_pairs_smoothing_and_batches(emu, seed)


def check_random_cross_wavelet_all_families(eng, seed=41):
    rs = np.random.RandomState(seed)
    for it in range(12):
        n = int(2 ** rs.uniform(4.5, 13))
        dt = float(10 ** rs.uniform(-1, 1))
        fam = int(rs.randint(3))
        par, mo = [(6.0, orc.Morlet(6)), (4, orc.Paul(4)), (2, orc.DOG(2))][fam]
        if rs.rand() < 0.3:
            par, mo = [(8.0, orc.Morlet(8)), (2, orc.Paul(2)), (5, orc.DOG(5))][fam]
        sj = (2 * dt / mo.flambda()) * 2 ** (np.arange(int(rs.randint(3, 20))) * 0.5)
        y1, y2 = rs.randn(n), rs.randn(n).cumsum()
        W12 = eng.xwt(y1, y2, dt, sj, fam, par)
        with np.errstate(all="ignore"):
            W1 = orc.cwt(y1, dt, wavelet=mo, freqs=1 / (mo.flambda() * sj))
            W2 = orc.cwt(y2, dt, wavelet=mo, freqs=1 / (mo.flambda() * sj))
        if W1[0].shape[0] != sj.size:      # Paul rows the reference drops: not the point here
            continue
        ref = W1[0] * W2[0].conj()
        check_rows(W12, ref, *ROW_GATE[0], what=(it, n, fam, par))


def test_random_cross_wavelet_all_families(emu):
    check_random_cross_wavelet_all_families(emu)
