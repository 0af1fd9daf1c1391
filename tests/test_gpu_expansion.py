"""The band-limited expansion path on the GPU, row by row.

Most rows of a long fp64 transform are written by the tensor-core expansion kernel
(kernels.cuh: ExpandMmaBody, fp64 mma.sync.m8n8k4): a coarse transform of Nc points expanded by
R = Np / Nc with a polyphase Kaiser-Bessel filter of 12, 16 or 20 taps.  The host-emulation
build runs neither that kernel nor the plans of the GPU planner (tap counts rounded to DMMA
k-steps, 20-tap coarse grids), so these tests cover it here: every tiling (R = 4, 8, 16, >= 32,
coarse grids shorter than one warp run, R = 2^14), both epilogues (store and the xwt
multiply-by-conjugate), odd lengths (scalar stores, the guarded last column), batched rows,
the scalar fp64 fallback and the alias-bound contract of set_expand_eps.

Each case compares every expansion row it fetches with the CPU oracle under the row-relative
gate of tests/_rowerr.py on white-noise input, and asserts its own coverage from last_plan()
(-log2 Nc per row) and from the kernel names of a profiled call, so that a planner change
cannot quietly empty it.  Worst row errors are printed (pytest -s)."""
import re

import numpy as np
import pytest

from _gpu_rows import fetch_rows, kernel_counts, oracle_rows, profiled
from _rowerr import check_rows
from oracle import cwt_oracle as orc

pytestmark = pytest.mark.gpu

# Row gate of the expansion rows (tests/_rowerr.py).  Measured on a B200 (1000 W power limit):
# worst row-relative error 5.2e-14 over every case of this file.  Zeroing the last tap of the
# tensor-core kernel's filter gives 2e-11 .. 1e-7 per row.
TOL_ROW = 1e-12
TOL_ABS = 1e-14
# Alias-bound contract: worst row error <= ALIAS_C * eps.  Measured on a B200: 7.7e-11 at eps 1e-6
# (12 taps), 2.6e-12 at 1e-9, 4.9e-14 at 5e-13 (0.1 eps: rounding, not aliasing, dominates there).
ALIAS_C = 1.0

MMA = re.compile(r"ExpandMmaBody<(\d+)(?:, (\d+))?>")
SCALAR64 = re.compile(r"ExpandBody<double, (\d+)(?:, (\d+))?>")
STORE, MULCONJ = 0, 1


@pytest.fixture(scope="module")
def eng():
    import pycwt_b200
    return pycwt_b200.default_engine()


def scales(log2N):
    """Quarter octaves from s = 32 (R = 8, 20 taps) to beyond the record (coarse grids of 64)."""
    return 2.0 ** (np.arange(20, 4 * (log2N + 2)) / 4.0)


def expand_kernels(prof, pattern=MMA):
    """{(taps, epilogue): launches} of the expansion kernels in a profile."""
    return kernel_counts(prof, pattern)


def expansion_rows(plan):
    return [i for i, p in enumerate(plan) if p < 0]


def factors(plan, log2N):
    """Expansion factors R = Np / Nc in the plan."""
    return {1 << (log2N + p) for p in plan if p < 0}


# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("log2N", [12, 14, 16, 20])
@pytest.mark.parametrize("length", ["Np", "Np-1", "Np/2+1", "Np-6"])
def test_tilings_and_lengths(eng, log2N, length):
    """Every tiling of ExpandMmaBody at one padded length: R = 8 (one warp across the phases),
    16 (two warps), 32 and more (four warps), coarse grids of 64 points (shorter than one warp
    run of 128: the warp-uniform early exit), R = 2^14 at Np = 2^20, rows of several coarse
    lengths in one launch (surplus tiles exit early).  Lengths: n0 = Np (paired 32-byte
    stores), odd n0 (row parity alternates: scalar stores on odd rows, the last column
    unpaired), n0 = Np/2 + 1 (most runs end past n0), n0 not a multiple of R."""
    Np = 1 << log2N
    n0 = {"Np": Np, "Np-1": Np - 1, "Np/2+1": Np // 2 + 1, "Np-6": Np - 6}[length]
    x = np.random.RandomState(log2N * 7 + len(length)).randn(n0)
    sj = scales(log2N)
    eng.cwt(x, 1.0, sj, 0, 6.0, fetch=False)
    plan = eng.last_plan(len(sj))
    rows = expansion_rows(plan)
    Rs = factors(plan, log2N)
    assert {8, 16, 32, Np // 64} <= Rs, sorted(Rs)
    if log2N == 20:
        assert -6 in plan and Np // 64 == 1 << 14, plan
    if log2N > 16:
        # the first and last row of each coarse length (the oracle's inverse FFTs cost)
        pick = set()
        for p in set(plan[i] for i in rows):
            r = [i for i in rows if plan[i] == p]
            pick.update((r[0], r[-1]))
        rows = sorted(pick)
    W = fetch_rows(eng, rows, n0)
    # the same transform profiled (streams serialised): bit-identical rows, and which kernels ran
    _, prof = profiled(eng, lambda: eng.cwt(x, 1.0, sj, 0, 6.0, fetch=False))
    assert np.array_equal(fetch_rows(eng, rows, n0), W)
    kern = expand_kernels(prof)
    if log2N == 12 and length == "Np":
        print("expansion kernels:", sorted(p["name"] for p in prof if "Expand" in p["name"]))
    assert set(kern) == {(12, STORE), (16, STORE), (20, STORE)}, prof
    assert not expand_kernels(prof, SCALAR64)
    # one launch per tap count: fewer launches than coarse lengths means a launch mixes them
    assert sum(kern.values()) < len(set(plan[i] for i in expansion_rows(plan))), (kern, plan)
    Wr = oracle_rows(x, sj, rows)
    err = check_rows(W, Wr, TOL_ROW, TOL_ABS, what=(log2N, n0))
    print("tilings Np=2^%d n0=%d: %d rows, R %s, worst row error %.2e"
          % (log2N, n0, len(rows), sorted(Rs), err))


def test_epilogues_at_odd_length(eng):
    """xwt (multiply-by-conjugate epilogue: read-modify-write of two adjacent points) and
    wct(sig=False) at an odd length, against the oracle; with the cwt of the same geometry all
    six instantiations ExpandMmaBody<12|16|20, store|mul-conj> run."""
    import pycwt_b200
    n0 = 8191
    rs = np.random.RandomState(77)
    y1, y2 = rs.randn(n0), rs.randn(n0)
    dj, s0, J = 0.25, 32.0, 40
    sj = s0 * 2 ** (np.arange(J + 1) * dj)
    W12, prof = profiled(eng, lambda: eng.xwt(y1, y2, 1.0, sj, 0, 6.0))
    rows = expansion_rows(eng.last_plan(len(sj)))
    assert rows
    # xwt = cwt of y1 (store) then cwt of y2 multiplied into it (mul-conj)
    kern = expand_kernels(prof)
    assert set(kern) >= {(12, MULCONJ), (16, MULCONJ), (20, MULCONJ)}, kern
    W12r = orc.xwt(y1, y2, 1.0, dj=dj, s0=s0, J=J, normalize=False)[0]
    err = check_rows(W12[rows], W12r[rows], TOL_ROW, TOL_ABS, what="xwt")
    print("xwt n0=%d: %d expansion rows, worst row error %.2e" % (n0, len(rows), err))
    _, prof = profiled(eng, lambda: eng.cwt(y1, 1.0, sj, 0, 6.0))
    stores = expand_kernels(prof)
    assert set(stores) == {(12, STORE), (16, STORE), (20, STORE)}, prof
    kern.update(stores)
    assert set(kern) == {(t, e) for t in (12, 16, 20) for e in (STORE, MULCONJ)}, kern
    # coherence: W1, W2 and W1 conj(W2) smoothed; the angle compared on the unit circle
    (WCT, aWCT, *_), prof = profiled(eng, lambda: pycwt_b200.wct(y1, y2, 1.0, dj=dj, s0=s0, J=J,
                                                                 sig=False))
    assert expand_kernels(prof)
    WCTr, aWCTr, *_ = orc.wct(y1, y2, 1.0, dj=dj, s0=s0, J=J, sig=False)
    err = check_rows(WCT, WCTr, TOL_ROW, TOL_ABS, what="wct")
    dang = np.abs(np.exp(1j * aWCT) - np.exp(1j * aWCTr)).max()
    print("wct n0=%d: worst row error %.2e, angle %.2e" % (n0, err, dang))
    assert dang < 1e-9


def test_batched_fp64_rows_odd_length(monkeypatch):
    """cwt_batch at odd n0 with an odd number of scales: the row index ch * S + j changes
    parity from one channel to the next (paired stores on some rows of a scale, scalar on
    others).  Bit-equal to per-channel transforms, in one chunk and in several."""
    from pycwt_b200 import _engine
    n0, S, nch = 8191, 13, 5
    rs = np.random.RandomState(5)
    X = rs.randn(nch, n0)
    sj = 2.0 ** (np.arange(20, 20 + 2 * S, 2) / 4.0)
    outs = []
    for mb in (None, "4"):                      # 4 MiB: two channels per chunk
        if mb:
            monkeypatch.setenv("CWTB_BATCH_MB", mb)
        e = _engine.Engine(0)
        try:
            _, W = e.cwt_batch(X, 1.0, sj, 0, 6.0, precision=0, want_power=False, want_w=True)
            for ch in range(nch):
                Wc = e.cwt(X[ch], 1.0, sj, 0, 6.0)
                assert np.array_equal(W[ch], Wc), (mb, ch)
            rows = expansion_rows(e.last_plan(S))
            assert len(rows) >= S - 2, rows
            _, prof = profiled(e, lambda: e.cwt_batch(X, 1.0, sj, 0, 6.0, precision=0,
                                                      want_power=False, want_w=True))
            assert expand_kernels(prof)
            outs.append(W)
        finally:
            e.close()
    assert np.array_equal(outs[0], outs[1])
    err = check_rows(outs[0][3], oracle_rows(X[3], sj, range(S)), TOL_ROW, TOL_ABS, what="batch")
    print("batched n0=%d S=%d: worst row error %.2e" % (n0, S, err))


def test_scalar_fp64_kernel(monkeypatch):
    """CWTB_EXPAND_MMA=0: the scalar ExpandBody<double, <= 16> and its own plan, same gate."""
    from pycwt_b200 import _engine
    monkeypatch.setenv("CWTB_EXPAND_MMA", "0")
    e = _engine.Engine(0)
    try:
        for n0 in (1 << 14, (1 << 14) - 1):
            x = np.random.RandomState(n0).randn(n0)
            sj = scales(14)
            W, prof = profiled(e, lambda: e.cwt(x, 1.0, sj, 0, 6.0))
            plan = e.last_plan(len(sj))
            rows = expansion_rows(plan)
            assert {8, 16, 32} <= factors(plan, 14), plan
            kern = expand_kernels(prof, SCALAR64)
            assert kern and max(t for t, _ in kern) <= 16 and not expand_kernels(prof), prof
            err = check_rows(W[rows], oracle_rows(x, sj, rows), TOL_ROW, TOL_ABS, what=n0)
            print("scalar fp64 kernel n0=%d: %d rows, taps %s, worst row error %.2e"
                  % (n0, len(rows), sorted(kern), err))
    finally:
        e.close()


def test_expansion_by_four_odd_lengths_and_xwt(monkeypatch):
    """R = 4 (CWTB_EXPAND_MIN_R=2): the tensor-core kernel's column layout of 2 coarse
    positions x 4 phases (B fragment shifted by one position), at odd lengths and through the
    multiply-by-conjugate epilogue."""
    from pycwt_b200 import _engine
    monkeypatch.setenv("CWTB_EXPAND_MIN_R", "2")
    e = _engine.Engine(0)
    sj = 2.0 * 2 ** (np.arange(8, 40) / 4.0)
    rs = np.random.RandomState(44)
    try:
        for n0 in ((1 << 14) - 1, (1 << 13) + 1, (1 << 14) - 6):
            x = rs.randn(n0)
            W, prof = profiled(e, lambda: e.cwt(x, 1.0, sj, 0, 6.0))
            plan = e.last_plan(len(sj))
            assert 4 in factors(plan, 14), plan
            assert expand_kernels(prof) and not expand_kernels(prof, SCALAR64), prof
            rows = expansion_rows(plan)
            err = check_rows(W[rows], oracle_rows(x, sj, rows), TOL_ROW, TOL_ABS, what=n0)
            print("R=4 cwt n0=%d: worst row error %.2e" % (n0, err))
        y2 = rs.randn(n0)
        W12, prof = profiled(e, lambda: e.xwt(x, y2, 1.0, sj, 0, 6.0))
        assert 4 in factors(e.last_plan(len(sj)), 14)
        assert MULCONJ in {ep for _, ep in expand_kernels(prof)}, prof
        ref = oracle_rows(x, sj, rows) * np.conj(oracle_rows(y2, sj, rows))
        err = check_rows(W12[rows], ref, TOL_ROW, TOL_ABS, what="xwt")
        print("R=4 xwt n0=%d: worst row error %.2e" % (n0, err))
    finally:
        e.close()


def test_alias_bound_contract(eng):
    """set_expand_eps(eps): every expansion row within ALIAS_C * eps of the oracle (the alias
    bound is a bound on the band spectrum; the l-infinity error can exceed it by up to the
    square root of the band's bins), and the loosest setting measurably worse than the
    tightest (the tap count reaches the kernel)."""
    n0 = 1 << 14
    x = np.random.RandomState(9).randn(n0)
    sj = scales(14)
    worst = {}
    try:
        for eps in (1e-6, 1e-9, 5e-13):
            eng.set_expand_eps(eps)
            W, prof = profiled(eng, lambda: eng.cwt(x, 1.0, sj, 0, 6.0))
            rows = expansion_rows(eng.last_plan(len(sj)))
            assert len(rows) > 20 and expand_kernels(prof)
            err = check_rows(W[rows], oracle_rows(x, sj, rows), ALIAS_C * eps, TOL_ABS, what=eps)
            worst[eps] = err
            print("expand eps %.0e: taps %s, worst row error %.2e (%.2f eps)"
                  % (eps, sorted(expand_kernels(prof)), err, err / eps))
    finally:
        eng.set_expand_eps()
    assert worst[1e-6] > 100 * worst[5e-13], worst


# ---- the randomised sweeps of tests/test_emu_stress.py on the GPU planner and kernels ----------
@pytest.mark.parametrize("seed,log2_max,draws", [(11, 15.5, 60), (12, 15.5, 60), (13, 15.5, 60),
                                                 (14, 20.0, 30)])
def test_random_transforms_gpu(eng, seed, log2_max, draws):
    from test_emu_stress import check_random_transforms
    checked, worst = check_random_transforms(eng, seed, log2_max, draws)
    print("seed %d: %d transforms, worst row error fp64 %.2e, fp32 %.2e"
          % (seed, checked, worst[0], worst[1]))
    assert checked > draws // 2


@pytest.mark.parametrize("seed", [31, 32])
def test_random_pairs_smoothing_and_batches_gpu(eng, seed):
    from test_emu_stress import check_random_pairs_smoothing_and_batches
    check_random_pairs_smoothing_and_batches(eng, seed)


def test_random_cross_wavelet_all_families_gpu(eng):
    from test_emu_stress import check_random_cross_wavelet_all_families
    check_random_cross_wavelet_all_families(eng)
