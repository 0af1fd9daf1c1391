"""The exact pruned-transform path row by row (CPU, host-emulation build; see
tests/test_emu_kernels.py for what that is).

Rows that do not take the band-limited expansion run through the exact kernels (kernels.cuh):
SingleBody<T, 32..1024> for K' <= 2^10, DirectBody<T, 2|4|8> for K' = 2^11..2^13, BandBody +
PassABody<T, K1, MODE_BAND> + PassBBody<T, +1, 512|1024> for the band two-kernel classes,
PassABody<T, K1, MODE_DENSE> (x^ psi^ generated in the kernel) for the dense scales, TinyBody for
Np < 32 and a pre-pass + interleaved 2^20-point transforms for Np > 2^20.

The cases are check_* functions that take an engine: this file runs them at Np <= 2^15 on the
emulation build, tests/test_gpu_exact.py runs them on the B200 up to Np = 2^22.  Each compares
every row it fetches with the CPU oracle under the row gate of tests/_rowerr.py on white noise,
and asserts its coverage from last_plan() (log2 K' per row, 0 for TinyBody) and, on the GPU,
from the kernel names of a profiled call, which must give bit-identical rows."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from _gpu_rows import fetch_rows, kernel_counts, oracle_rows, profiled
from _rowerr import check_rows
from oracle import cwt_oracle as orc

# Row gates (tests/_rowerr.py) per engine precision: (tol_row, tol_abs).  Measured worst row
# errors are in tests/test_gpu_exact.py.
GATE = {0: (1e-13, 1e-15), 1: (2e-6, 1e-7)}

# engine family id, parameter, oracle mother.  DOG: negative-frequency residues (rsplit, the
# negative-row twist), odd orders have an imaginary unit; order 10 is evaluated in double by the
# fp32 kernels (band_value).  Paul: one-sided band, the window is widened to contain k = 0.
FAMILIES = {
    "morlet": (0, 6.0, orc.Morlet(6)),
    "dog2": (2, 2, orc.DOG(2)),
    "dog3": (2, 3, orc.DOG(3)),
    "dog10": (2, 10, orc.DOG(10)),
    "paul4": (1, 4, orc.Paul(4)),
}
# one sampling interval per family: the band limits and fam.dw depend on it
DT = {"morlet": 1.0, "dog2": 0.25, "dog3": 0.25, "dog10": 2.0, "paul4": 3.0}

DENSE, BAND, CPLX = 0, 1, 3          # kernels.cuh: MODE_DENSE, MODE_BAND, MODE_CPLX
EXACT = re.compile(r"^(SingleBody|DirectBody|PassABody|PassBBody|TinyBody)<(double|float)"
                   r"(?:, (-?\d+))?(?:, (-?\d+))?(?:, (-?\d+))?>")


@pytest.fixture(scope="module")
def emu_lib():
    from pycwt_b200 import build as _build
    return _build.build_emulation(os.path.join(ROOT, "tests", "_emu"))


@pytest.fixture(scope="module")
def emu(emu_lib):
    from pycwt_b200 import _engine
    eng = _engine.Engine(0, lib_path=emu_lib)
    yield eng
    eng.close()


def emulated(eng):
    """The emulation build runs every launch in order and records no profile."""
    return "emulation" in eng.version()


def exact_kernels(prof):
    """Exact-path kernels of a profile (the forward FFT, tagged "fwd:", is left out):
    ("SingleBody", T, K), ("DirectBody", T, K1), ("PassABody", T, K1, MODE),
    ("PassBBody", T, K2), ("TinyBody", T)."""
    out = set()
    for (kind, T, a, b, c) in kernel_counts(prof, EXACT, default=None):
        if kind in ("SingleBody", "DirectBody"):
            out.add((kind, T, a))
        elif kind == "PassABody":
            out.add((kind, T, a, b))
        elif kind == "PassBBody":              # <T, SIGN, K2>: K2 = K2C = 1024 is the default
            out.add((kind, T, b or 1024))
        else:
            out.add((kind, T))
    return out


def test_kernel_name_parser():
    """exact_kernels() on names as the engine's profile reports them (engine.cu: body_name), with
    and without the defaulted second-pass length; the forward transform's launches are left out."""
    names = ["SingleBody<double, 256>", "DirectBody<float, 4>", "PassABody<double, 16, 1, 1>",
             "PassABody<float, 1024, 0, 1>", "PassBBody<double, 1, 512>", "PassBBody<double, 1, 1024>",
             "PassBBody<float, 1>", "TinyBody<double>", "TinyFwdBody<double>", "BandBody<double>",
             "fwd:PassABody<double, 32, 2, -1>", "fwd:PassBBody<double, -1, 1024>",
             "ExpandMmaBody<12, 1>"]
    prof = [{"name": n, "launches": 1, "ms": 0.0, "rows": 1} for n in names]
    assert exact_kernels(prof) == {
        ("SingleBody", "double", 256), ("DirectBody", "float", 4),
        ("PassABody", "double", 16, BAND), ("PassABody", "float", 1024, DENSE),
        ("PassBBody", "double", 512), ("PassBBody", "double", 1024), ("PassBBody", "float", 1024),
        ("TinyBody", "double")}


def expected_kernels(plan, log2N, T, direct_max=13, k2_band=9, k2_512_max=16):
    """The kernels the planner's classes launch (engine.cu: run_job), from last_plan()."""
    out = set()
    for lk in set(plan):
        if lk == 0:
            out.add(("TinyBody", T))
        elif lk <= 10:
            out.add(("SingleBody", T, 1 << lk))
        elif lk <= direct_max and lk < log2N:
            out.add(("DirectBody", T, 1 << (lk - 10)))
        elif lk == log2N and log2N > 20:             # pre-pass, then interleaved 2^20-point rows
            out |= {("PassABody", T, 1 << (log2N - 20), DENSE), ("PassABody", T, 1024, CPLX),
                    ("PassBBody", T, 1024)}
        elif lk == log2N:
            out |= {("PassABody", T, 1 << (log2N - 10), DENSE), ("PassBBody", T, 1024)}
        else:
            # fp32 always takes the 1024-point second pass (its 512-point tile rows are not
            # 16-byte aligned), and so does a first kernel whose tile of 4096 points spans more
            # than 512 values of r2 (K1 < 8)
            l2k = 10 if (T == "float" or lk > k2_512_max or lk - k2_band < 3) else k2_band
            out |= {("PassABody", T, 1 << (lk - l2k), BAND), ("PassBBody", T, 1 << l2k)}
    return out


def expected_classes(log2N, dense_margin=2, fam="morlet"):
    """Every class a scale sweep from below Nyquist to beyond the record meets at Np = 2^log2N:
    pruned lengths 2^5 .. 2^(log2N-1) (those of 2^18 or more within dense_margin octaves of Np
    run as dense scales, below Np = 2^21) and the dense class.  A one-sided band (Paul) spans
    Np/2 bins at most: dense only through that promotion."""
    if log2N < 5:
        return {0}
    band = set(range(5, min(log2N, 21)))
    promoted = {lk for lk in band if lk >= 18 and log2N <= 20 and log2N - lk <= dense_margin}
    dense = {log2N} if (promoted or not fam.startswith("paul")) else set()
    return (band - promoted) | dense


def sweep_scales(log2N, dt):
    """Quarter octaves from s = dt / 2 (band beyond Nyquist: dense) to 4 Np dt (beyond the record:
    K' = 32)."""
    return dt * 2.0 ** (np.arange(-4, 4 * (log2N + 2) + 1) / 4.0)


def lengths(log2N):
    """n0 = Np (unguarded stores), Np - 1 (odd: the guarded last column), Np/2 + 1 (most of the
    second half trimmed) and Np - 6 (not a multiple of the store width)."""
    Np = 1 << log2N
    return {"Np": Np, "Np-1": Np - 1, "Np/2+1": Np // 2 + 1, "Np-6": Np - 6}


def class_ends(plan, rows=None):
    """The first and the last row of each class."""
    rows = range(len(plan)) if rows is None else rows
    pick = set()
    for p in set(plan[i] for i in rows):
        r = [i for i in rows if plan[i] == p]
        pick.update((r[0], r[-1]))
    return sorted(pick)


def finite_rows(Wr):
    """Rows the reference computes (Paul: inf * 0 at large negative frequencies gives NaN)."""
    return np.isfinite(Wr).all(axis=1)


def run_checked(eng, x, dt, sj, fam, prec, rows, expect=None, oracle=None):
    """Exact-mode transform of x, rows `rows` fetched, profiled again (bit-identical rows, the
    kernel names against `expect(plan)`), and compared with the oracle under the row gate.
    Returns (worst row error, plan, rows, kernels seen)."""
    fid, par, mo = FAMILIES[fam]
    n0 = len(x)
    eng.cwt(x, dt, sj, fid, par, prec, fetch=False)
    plan = eng.last_plan(len(sj))
    rows = rows(plan) if callable(rows) else rows
    W = fetch_rows(eng, rows, n0)
    seen = set()
    if not emulated(eng):
        _, prof = profiled(eng, lambda: eng.cwt(x, dt, sj, fid, par, prec, fetch=False))
        assert np.array_equal(fetch_rows(eng, rows, n0), W), "profiled call differs"
        seen = exact_kernels(prof)
        if expect is not None:
            assert seen == expect(plan), (sorted(seen), sorted(expect(plan)), plan)
    Wr = oracle(rows) if oracle else oracle_rows(x, sj, rows, mo, dt)
    ok = finite_rows(Wr)
    err = check_rows(W[ok], Wr[ok], *GATE[prec], what=(fam, n0, prec))
    return err, plan, rows, seen


# ---- 1, 2: every class at every padded length, both precisions ----------------------------------
def check_every_class(eng, log2N, length, fam, prec=0, all_rows=True):
    """Exact mode at Np = 2^log2N: every class, the oracle on every row (all_rows) or on the first
    and the last row of each class.  Returns (worst row error, kernels seen)."""
    n0 = lengths(log2N)[length]
    dt = DT[fam]
    rs = np.random.RandomState(1000 * log2N + 10 * len(length) + len(fam) + prec)
    x = rs.randn(n0)
    if prec:
        x = x.astype(np.float32)
    sj = sweep_scales(log2N, dt)
    T = "float" if prec else "double"
    eng.set_expand_eps(0.0, 0.0)
    try:
        err, plan, rows, seen = run_checked(
            eng, x, dt, sj, fam, prec, (lambda p: list(range(len(p)))) if all_rows else class_ends,
            expect=lambda p: expected_kernels(p, log2N, T))
    finally:
        eng.set_expand_eps()
    assert set(plan) == expected_classes(log2N, fam=fam), (sorted(set(plan)), fam, log2N)
    return err, seen


@pytest.mark.parametrize("log2N", [11, 12, 13, 14, 15])
def test_every_class_emulated(emu, log2N):
    worst = {0: 0.0, 1: 0.0}
    for i, length in enumerate(lengths(log2N)):
        for fam in ("morlet", "dog2" if i % 2 else "dog3", "paul4"):
            worst[0] = max(worst[0], check_every_class(emu, log2N, length, fam)[0])
        fam32 = ("morlet", "dog10", "dog3", "paul4")[i]
        worst[1] = max(worst[1], check_every_class(emu, log2N, length, fam32, prec=1)[0])
    print("Np=2^%d: worst row error fp64 %.2e, fp32 %.2e" % (log2N, worst[0], worst[1]))


# ---- 4: kernel-choice switches --------------------------------------------------------------
# (environment, planner arguments of expected_kernels, the kernel that must appear)
SWITCHES = [
    ({"CWTB_DIRECT_MAX": "10"}, {"direct_max": 10}, ("PassABody", "double", 2, BAND)),
    ({"CWTB_DIRECT_MAX": "11"}, {"direct_max": 11}, ("PassABody", "double", 8, BAND)),
    ({"CWTB_DIRECT_MAX": "12"}, {"direct_max": 12}, ("PassABody", "double", 16, BAND)),
    ({"CWTB_K2_BAND": "10"}, {"k2_band": 10}, ("PassABody", "double", 16, BAND)),
    ({"CWTB_K2_512_MAX": "13"}, {"k2_512_max": 13}, ("PassABody", "double", 16, BAND)),
    ({"CWTB_K2_512_MAX": "19"}, {"k2_512_max": 19}, ("PassABody", "double", 256, BAND)),
]


def check_kernel_switches(make_engine, monkeypatch, log2N, settings=SWITCHES, fam="morlet", seen=None):
    """One exact-mode geometry with every class at Np = 2^log2N (n0 odd) under each setting of a
    kernel-choice switch, on a new engine each (switches are read when a context is created).
    Oracle rows are computed once and shared.  Returns {setting: worst row error}; the kernels
    launched are added to `seen`."""
    n0 = (1 << log2N) - 3
    dt = DT[fam]
    x = np.random.RandomState(log2N).randn(n0)
    sj = sweep_scales(log2N, dt)
    mo = FAMILIES[fam][2]
    cache = {}

    def oracle(rows):
        need = [j for j in rows if j not in cache]
        for j, r in zip(need, oracle_rows(x, sj, need, mo, dt)):
            cache[j] = r
        return np.array([cache[j] for j in rows])

    pick = class_ends if log2N > 16 else (lambda p: list(range(len(p))))
    seen_all = seen
    out = {}
    base = None
    for env, args, marker in [({}, {}, None)] + list(settings):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = make_engine()
        try:
            e.set_expand_eps(0.0, 0.0)
            err, plan, rows, seen = run_checked(
                e, x, dt, sj, fam, 0, pick, oracle=oracle,
                expect=lambda p: expected_kernels(p, log2N, "double", **args))
        finally:
            e.close()
            for k in env:
                monkeypatch.delenv(k)
        key = " ".join("%s=%s" % kv for kv in env.items()) or "default"
        margin = int(env.get("CWTB_DENSE_MARGIN", 2))
        assert set(plan) == expected_classes(log2N, margin, fam), (key, sorted(set(plan)))
        if seen_all is not None:
            seen_all |= seen
        if base is None:
            base = seen
        elif seen:       # the switch reached the planner: the launched kernels changed as it claims
            assert marker in seen and marker not in base and seen != base, (key, sorted(seen))
        out[key] = err
    return out


def test_kernel_switches_emulated(emu_lib, monkeypatch):
    from pycwt_b200 import _engine
    worst = check_kernel_switches(lambda: _engine.Engine(0, lib_path=emu_lib), monkeypatch, 15)
    for k, v in worst.items():
        print("Np=2^15 %s: worst row error %.2e" % (k, v))


# ---- 6: batched exact rows --------------------------------------------------------------------
def check_batched_exact(make_engine, monkeypatch, log2N, nch, mbs=(None,)):
    """cwt_batch in exact mode at odd n0, fp64 and fp32, in one chunk and in several
    (CWTB_BATCH_MB): rows bit-equal to per-channel cwt (the channel offset d.chan * N in
    band_value and in the dense generator), one channel against the oracle."""
    n0 = (1 << log2N) - 1
    rs = np.random.RandomState(log2N + nch)
    X = rs.randn(nch, n0)
    fam = "dog3"
    fid, par, mo = FAMILIES[fam]
    dt = DT[fam]
    sj = sweep_scales(log2N, dt)[::2]
    worst = {0: 0.0, 1: 0.0}
    results = {}
    for mb in mbs:
        if mb:
            monkeypatch.setenv("CWTB_BATCH_MB", mb)
        e = make_engine()
        try:
            e.set_expand_eps(0.0, 0.0)
            for prec in (0, 1):
                Xp = X.astype(np.float32) if prec else X
                _, W = e.cwt_batch(Xp, dt, sj, fid, par, precision=prec, want_power=False, want_w=True)
                for ch in range(nch):
                    Wc = e.cwt(Xp[ch], dt, sj, fid, par, prec, out_f64=False)
                    assert np.array_equal(W[ch], Wc), (mb, prec, ch)
                assert set(e.last_plan(len(sj))) == expected_classes(log2N, fam=fam), e.last_plan(len(sj))
                results.setdefault(prec, []).append(W)
                ch = nch // 2
                Wr = oracle_rows(Xp[ch], sj, range(len(sj)), mo, dt)
                ok = finite_rows(Wr)
                worst[prec] = max(worst[prec], check_rows(W[ch][ok], Wr[ok], *GATE[prec],
                                                          what=("batch", mb, prec)))
        finally:
            e.close()
            if mb:
                monkeypatch.delenv("CWTB_BATCH_MB")
    for prec, Ws in results.items():
        assert all(np.array_equal(Ws[0], w) for w in Ws[1:]), prec
    return worst


def test_batched_exact_emulated(emu_lib, monkeypatch):
    from pycwt_b200 import _engine
    worst = check_batched_exact(lambda: _engine.Engine(0, lib_path=emu_lib), monkeypatch, 12, 3)
    print("batched: worst row error fp64 %.2e, fp32 %.2e" % (worst[0], worst[1]))


# ---- 7: tiny and small transforms -----------------------------------------------------------------
TINY_AND_SMALL = (5, 9, 16, 17, 31, 32, 33, 100, 255, 256, 257, 600, 1023, 1024)


def check_tiny_and_small(eng):
    """n0 = 5, 9, 16 (TinyBody, Np < 32) and n0 = 17 .. 1024 (Np = 32 .. 1024: single-kernel
    classes only), every family, both precisions.  Returns {precision: worst row error}."""
    worst = {0: 0.0, 1: 0.0}
    seen = set()
    for n0 in TINY_AND_SMALL:
        log2N = max(1, int(np.ceil(np.log2(n0))))
        for fam in ("morlet", "dog2", "dog3", "paul4"):
            for prec in (0, 1):
                x = np.random.RandomState(n0).randn(n0)
                if prec:
                    x = x.astype(np.float32)
                sj = sweep_scales(log2N, DT[fam])
                T = "float" if prec else "double"
                eng.set_expand_eps(0.0, 0.0)
                try:
                    err, plan, _, s = run_checked(eng, x, DT[fam], sj, fam, prec, list(range(len(sj))),
                                                  expect=lambda p: expected_kernels(p, log2N, T))
                finally:
                    eng.set_expand_eps()
                if log2N < 5:
                    assert set(plan) == {0}, plan
                else:
                    assert set(plan) == set(range(5, log2N + 1)) - (
                        {log2N} if fam == "paul4" and log2N > 5 else set()), (n0, fam, plan)
                worst[prec] = max(worst[prec], err)
                seen |= s
    return worst, seen


def test_tiny_and_small_emulated(emu):
    worst, _ = check_tiny_and_small(emu)
    print("tiny and small: worst row error fp64 %.2e, fp32 %.2e" % (worst[0], worst[1]))
