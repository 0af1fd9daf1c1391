"""The exact pruned-transform path on the GPU, row by row.

The cases of tests/test_emu_exact.py (every class at every padded length, both precisions,
the kernel-choice switches, batched rows, tiny and small transforms) on the B200 up to Np = 2^22,
and what only the GPU has: the streams, chains and chunks of the two-kernel classes (their
schedule switches must give bit-identical W), the bulk-async row loads of PassBBody and the
three-level path beyond 2^20.  Every fetched exact row is compared with the CPU oracle under the
row gate of tests/_rowerr.py on white noise; each case asserts its coverage from last_plan() and
from the kernel names of a profiled call (streams serialised, rows bit-identical).  Worst row
errors are printed (pytest -s).

Gates (test_emu_exact.GATE): fp64 1e-13 per row (+ 1e-15 of max|W|), fp32 2e-6 (+ 1e-7).
Worst row-relative errors measured on the emulation build (same kernel sources, Np <= 2^15):
fp64 5.5e-15, fp32 1.0e-6.  Not yet measured on a B200; the fp32 gate is within 2x of the
emulated figure, so a B200 figure above it needs explaining before the gate moves."""
import numpy as np
import pytest

from _gpu_rows import oracle_rows, profiled
from _rowerr import check_rows
from test_emu_exact import (BAND, DENSE, DT, GATE, check_batched_exact, check_every_class,
                            check_kernel_switches, check_tiny_and_small, class_ends, emulated,
                            exact_kernels, expected_classes, expected_kernels, run_checked,
                            sweep_scales)

pytestmark = pytest.mark.gpu

SEEN = set()      # exact-path kernels launched by the cases of this file


@pytest.fixture(scope="module")
def eng():
    import pycwt_b200
    return pycwt_b200.default_engine()


def new_engine():
    from pycwt_b200 import _engine
    return _engine.Engine(0)


# ---- 1, 2: every class at every padded length, both precisions --------------------------------
@pytest.mark.parametrize("log2N", list(range(11, 21)))
@pytest.mark.parametrize("length", ["Np", "Np-1", "Np/2+1", "Np-6"])
def test_every_class(eng, log2N, length):
    """Single 2^5..2^10, direct 2^11..2^13, band 2^14..2^17 (512-point second pass up to 2^16,
    1024 at 2^17) and dense K1 = Np / 1024, for Morlet, DOG and Paul at dt != 1; at 2^20 the
    first and last row of each class only."""
    i = ["Np", "Np-1", "Np/2+1", "Np-6"].index(length)
    fams = ("morlet", "dog2" if i % 2 else "dog3", "paul4")
    if log2N >= 18:                  # bound the oracle's cost: one family per length
        fams = (("morlet", "dog3", "paul4", "dog2")[i],)
    worst = 0.0
    for fam in fams:
        err, seen = check_every_class(eng, log2N, length, fam, all_rows=log2N < 20)
        SEEN.update(seen)
        worst = max(worst, err)
    print("fp64 Np=2^%d n0=%s %s: worst row error %.2e" % (log2N, length, fams, worst))


@pytest.mark.parametrize("log2N", list(range(11, 21)))
@pytest.mark.parametrize("length", ["Np-1", "Np-6"])
def test_every_class_fp32(eng, log2N, length):
    """The fp32 engine on a float32 signal: every band class with the 1024-point second pass
    (PassABody<float, 16, MODE_BAND> at K' = 2^14), DOG of order 10 (amplitude in double) and of
    order 3 (in float)."""
    fams = ("dog10", "paul4") if length == "Np-1" else ("morlet", "dog3")
    worst = 0.0
    for fam in fams:
        err, seen = check_every_class(eng, log2N, length, fam, prec=1, all_rows=log2N < 20)
        SEEN.update(seen)
        worst = max(worst, err)
    if log2N >= 15:                  # K' = 2^14 is a band class from Np = 2^15 on
        assert ("PassABody", "float", 16, BAND) in seen, sorted(seen)
    print("fp32 Np=2^%d n0=%s %s: worst row error %.2e" % (log2N, length, fams, worst))


# ---- 3: Np > 2^20 ------------------------------------------------------------------------------
@pytest.mark.parametrize("n0", [2 ** 20 + 4321, 2 ** 21 - 1, 2 ** 22 - 5])
def test_beyond_2_20(eng, n0):
    """Np = 2^21, 2^22: the three-level dense path (a PassABody<double, Np / 2^20, MODE_DENSE>
    pre-pass, then 2^20-point transforms with interleaved stores) and band classes 2^18..2^20
    (K1 = 256, 512, 1024 with the 1024-point second pass).  Selected rows only."""
    log2N = int(np.ceil(np.log2(n0)))
    x = np.random.RandomState(n0 % 1000).randn(n0)
    fam = "morlet" if n0 & 1 else "dog2"
    dt = DT[fam]
    sj = dt * 2.0 ** (np.arange(-4, 4 * (log2N + 2) + 1, 2) / 4.0)
    eng.set_expand_eps(0.0, 0.0)
    try:
        err, plan, rows, seen = run_checked(
            eng, x, dt, sj, fam, 0, lambda p: class_ends(p, [i for i in range(len(p)) if p[i] >= 14]),
            expect=lambda p: expected_kernels(p, log2N, "double"))
    finally:
        eng.set_expand_eps()
    SEEN.update(seen)
    assert set(plan) == expected_classes(log2N), sorted(set(plan))
    assert {("PassABody", "double", 1 << (log2N - 20), DENSE), ("PassABody", "double", 1024, BAND),
            ("PassABody", "double", 256, BAND)} <= seen, sorted(seen)
    print("Np=2^%d n0=%d: %d rows, worst row error %.2e" % (log2N, n0, len(rows), err))


# ---- 4: kernel-choice switches ---------------------------------------------------------------------
def test_kernel_switches(monkeypatch):
    """CWTB_DIRECT_MAX (2^11..2^13 from DirectBody to band K1 = 2, 8, 16), CWTB_K2_BAND=10,
    CWTB_K2_512_MAX = 13 and 19, against the oracle at Np = 2^18; CWTB_DENSE_MARGIN=0 at 2^20
    (band K1 = 256, 512).  Each must change the launched kernels as it claims."""
    worst = check_kernel_switches(new_engine, monkeypatch, 18, seen=SEEN)
    worst.update(check_kernel_switches(
        new_engine, monkeypatch, 20, seen=SEEN,
        settings=[({"CWTB_DENSE_MARGIN": "0"}, {}, ("PassABody", "double", 512, BAND))]))
    for k, v in worst.items():
        print("switch %s: worst row error %.2e" % (k, v))


def test_gauss_recurrence_against_exp(monkeypatch):
    """Dense Morlet rows with the Gaussian by recurrence (default) and by exp per bin
    (CWTB_GAUSS_REC=0): both under the row gate, and their worst row difference reported."""
    log2N = 20
    n0 = (1 << log2N) - 1
    x = np.random.RandomState(3).randn(n0)
    sj = 2.0 ** (np.arange(-4, 8) / 4.0)            # dense at Np = 2^20
    out = {}
    for rec in ("1", "0"):
        monkeypatch.setenv("CWTB_GAUSS_REC", rec)
        e = new_engine()
        try:
            e.set_expand_eps(0.0, 0.0)
            W, prof = profiled(e, lambda: e.cwt(x, 1.0, sj, 0, 6.0))
            assert set(e.last_plan(len(sj))) == {log2N}
            assert ("PassABody", "double", 1024, DENSE) in exact_kernels(prof)
            out[rec] = np.array(W)
            del W
        finally:
            e.close()
    monkeypatch.delenv("CWTB_GAUSS_REC")
    Wr = oracle_rows(x, sj, range(len(sj)))
    errs = {rec: check_rows(W, Wr, *GATE[0], what=rec) for rec, W in out.items()}
    d = np.abs(out["1"] - out["0"]).max(axis=1) / np.abs(out["0"]).max(axis=1)
    assert not np.array_equal(out["1"], out["0"])     # the switch reaches the kernel
    print("dense Morlet: worst row error recurrence %.2e, exp %.2e; worst row difference %.2e"
          % (errs["1"], errs["0"], d.max()))


# ---- 5: schedule switches: bit-identical W ----------------------------------------------------------
SCHEDULES = [
    {"CWTB_STREAMS": "1"}, {"CWTB_STREAMS": "2"}, {"CWTB_STREAMS": "3"},
    {"CWTB_CHAINS": "1"}, {"CWTB_CHAINS": "2"}, {"CWTB_CHAINS": "4"},
    {"CWTB_GROUP": "1"}, {"CWTB_GROUP": "0"}, {"CWTB_GROUP": "0", "CWTB_GROUP_MB": "40"},
    {"CWTB_PASSB_REV": "0"},
    {"CWTB_PF_DIST": "0", "CWTB_PF_DIST_A": "0"},
    {"CWTB_PRIO": "0"}, {"CWTB_PRIO": "2"}, {"CWTB_PRIO_FAN": "1"}, {"CWTB_PRIO_FAN": "8"},
    {"CWTB_PLAN_REUSE": "0"},
]


def test_schedule_switches_bit_identical(monkeypatch):
    """One transform at Np = 2^20, odd n0, chunks of three rows (CWTB_GROUP=3), once in exact
    mode (every exact class) and once in the default mode (exact and expansion rows together),
    repeated under every schedule switch and profiled: every row equal to the reference run bit
    for bit.  The arithmetic of a row does not depend on the stream, chain, chunk or order it
    runs in, so any difference is a race."""
    log2N = 20
    n0 = (1 << log2N) - 3
    x = np.random.RandomState(55).randn(n0)
    sj = sweep_scales(log2N, 1.0)[::2]
    monkeypatch.setenv("CWTB_GROUP", "3")

    def run(e):
        out = []
        for eps in ((0.0, 0.0), ()):
            e.set_expand_eps(*eps)
            W = e.cwt(x, 1.0, sj, 0, 6.0)
            out.append((np.array(W), e.last_plan(len(sj))))
            W = e.cwt(x, 1.0, sj, 0, 6.0)             # the same call again (plan reuse)
            assert np.array_equal(W, out[-1][0])
            del W
        e.set_expand_eps()
        return out

    e = new_engine()
    try:
        ref = run(e)
        prof_run = profiled(e, lambda: run(e))[0]
    finally:
        e.close()
    (W_exact, plan_exact), (W_def, plan_def) = ref
    assert set(plan_exact) == expected_classes(log2N), sorted(set(plan_exact))
    assert min(plan_def) < 0 and max(plan_def) == log2N, sorted(set(plan_def))
    assert any(14 <= p < log2N for p in plan_def), sorted(set(plan_def))   # exact band rows too
    # the reference run itself against the oracle on the first and last row of each class
    rows = class_ends(plan_exact)
    check_rows(W_exact[rows], oracle_rows(x, sj, rows), *GATE[0], what="schedule reference")
    differ = []

    def compare(key, got):
        for (W, plan), (Wref, pref) in zip(got, ref):
            assert plan == pref, key
            bad = np.nonzero([not np.array_equal(a, b) for a, b in zip(W, Wref)])[0]
            if bad.size:
                differ.append((key, bad.tolist(), [plan[i] for i in bad]))

    compare("profiled", prof_run)
    for env in SCHEDULES:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = new_engine()
        try:
            compare(env, run(e))
        finally:
            e.close()
            for k in env:
                if k == "CWTB_GROUP":
                    monkeypatch.setenv(k, "3")
                else:
                    monkeypatch.delenv(k)
    assert not differ, differ
    print("schedule switches: %d settings bit-identical to the reference" % (len(SCHEDULES) + 1))


# ---- 6: batched exact rows ---------------------------------------------------------------------------
def test_batched_exact(monkeypatch):
    """cwt_batch in exact mode at odd n0, fp64 and fp32, five channels in one chunk and in several
    (CWTB_BATCH_MB=80: chunks of two channels in fp64, of four in fp32)."""
    worst = check_batched_exact(new_engine, monkeypatch, 16, 5, mbs=(None, "80"))
    print("batched: worst row error fp64 %.2e, fp32 %.2e" % (worst[0], worst[1]))


# ---- 7: tiny and small ---------------------------------------------------------------------------------
def test_tiny_and_small(eng):
    worst, seen = check_tiny_and_small(eng)
    SEEN.update(seen)
    if not emulated(eng):
        assert {("TinyBody", "double"), ("TinyBody", "float")} <= seen
    print("tiny and small: worst row error fp64 %.2e, fp32 %.2e" % (worst[0], worst[1]))


def test_union_of_kernels():
    """Every exact-path instantiation of cwt ran in this file (when the whole file ran)."""
    if len(SEEN) < 10:
        pytest.skip("the other cases of this file did not run")
    want = set()
    for T in ("double", "float"):
        want |= {("SingleBody", T, 1 << k) for k in range(5, 11)}
        want |= {("DirectBody", T, k) for k in (2, 4, 8)}
        want |= {("PassABody", T, 1 << k, DENSE) for k in range(1, 11)}
        want |= {("TinyBody", T), ("PassBBody", T, 1024)}
    want |= {("PassABody", "double", k, BAND) for k in (32, 64, 128, 256, 512, 1024)}
    want |= {("PassABody", "double", k, BAND) for k in (2, 8, 16)}
    want |= {("PassABody", "float", k, BAND) for k in (16, 32, 64, 128)}
    want.add(("PassBBody", "double", 512))
    missing = want - SEEN
    assert not missing, sorted(missing)
