"""cwt_batch's per-channel products on the B200 (BatchProductsBody in the pipelined chunk loop).

The checks are those of tests/test_emu_batch_products.py, at sizes the emulation build cannot
reach: config 5's geometry with fewer channels (fp32, n0 = 2^16, S = 128) and long fp64 rows
(n0 = 2^18, S = 64), where both the expansion rows and the exact two-kernel rows are present.
Gates: max|diff| / max|ref| per channel and product (GATES there)."""
import numpy as np
import pytest

from _gpu_rows import kernel_counts, profiled
from test_emu_batch_products import (check_batch_products, check_errors, check_products_subsets,
                                     white)

pytestmark = pytest.mark.gpu


def new_engine():
    from pycwt_b200 import _engine
    return _engine.Engine(0)


def show(what, worst):
    print(what, {"%s/%s" % k: "%.1e" % v for k, v in sorted(worst.items())})


def test_config5_geometry_fp32(monkeypatch):
    # 64 channels in chunks of 7 (the last one holds 1)
    w = check_batch_products(new_engine, monkeypatch, "morlet_c5", 1 << 16, "fp32", nch=64, seed=11,
                             mb=7 * 64, oracle_channels=[0, 6, 7, 63])
    show("fp32 64 x 2^16 S=128:", w)


def test_long_rows_fp64(monkeypatch):
    # 4 channels in chunks of 3 and 1; expansion rows and exact two-kernel rows
    from pycwt_b200 import _engine
    e = new_engine()
    try:
        import pycwt_b200 as pycwt
        sj, _ = pycwt.batch._resolve_scales(1 << 18, 1.0, 1 / 4, 2, 63, pycwt.Morlet(6), None)
        e.cwt(white(1, 1 << 18, 0)[0], 1.0, sj, _engine.MORLET, 6.0, _engine.F64, fetch=False)
        plan = e.last_plan(len(sj))
        assert min(plan) < 0 and max(plan) > 13, plan      # expansion rows; two-kernel exact rows
    finally:
        e.close()
    w = check_batch_products(new_engine, monkeypatch, "morlet_s64", 1 << 18, "fp64", nch=4, seed=12,
                             mb=3 * 256 + 1, oracle_channels=[0, 3])
    show("fp64 4 x 2^18 S=64:", w)


def test_subsets_and_errors(monkeypatch):
    check_products_subsets(new_engine, monkeypatch)
    check_products_subsets(new_engine, monkeypatch, n0=4096, prec="fp32")
    check_errors(new_engine, monkeypatch)


def _products_call(e, X, sj, nbands=2, f32=True):
    from pycwt_b200 import _engine
    S = sj.size
    lo = np.full(S, X.shape[1] // 4, dtype=np.int64)
    hi = np.full(S, 3 * X.shape[1] // 4, dtype=np.int64)
    wt = np.random.RandomState(1).rand(nbands, S)
    return e.cwt_batch_products(X, 1.0, sj, _engine.MORLET, 6.0, _engine.F32 if f32 else _engine.F64,
                                coi_ranges=(lo, hi), band_weights=wt,
                                chan_scale=np.linspace(1, 2, X.shape[0]), icwt_factor=0.3 + 0.1j)


@pytest.mark.parametrize("nbands,f32", [(2, True), (8, True), (2, False), (8, False)])
def test_pipelined_matches_chunk_after_chunk(monkeypatch, nbands, f32):
    """Column outputs are written without atomics: bit-identical between the two chunk loops."""
    X = white(16, 1 << 16, 21, f32)
    sj = 2.0 * 2 ** (np.arange(128) / 8)
    monkeypatch.setenv("CWTB_BATCH_MB", "200")          # chunks of 3 (fp32) / 1 (fp64) channels
    out = {}
    for pipe in ("1", "0"):
        monkeypatch.setenv("CWTB_BATCH_PIPELINE", pipe)
        e = new_engine()
        try:
            out[pipe] = [None if a is None else np.array(a) for a in _products_call(e, X, sj, nbands, f32)]
        finally:
            e.close()
    (p1, c1, b1, i1), (p0, c0, b0, i0) = out["1"], out["0"]
    assert np.array_equal(b1, b0) and np.array_equal(i1, i0)
    np.testing.assert_allclose(p1, p0, rtol=1e-12)
    np.testing.assert_allclose(c1, c0, rtol=1e-12)


def test_profiled_launches(monkeypatch):
    """A products call launches one BatchProductsBody per chunk and no PowerBody; the
    spectra-only cwt_batch still launches PowerBody (one per chunk)."""
    from pycwt_b200 import _engine
    X = white(16, 1 << 16, 22, True)
    sj = 2.0 * 2 ** (np.arange(128) / 8)
    monkeypatch.setenv("CWTB_BATCH_MB", "200")          # 3 channels per chunk: 6 chunks
    e = new_engine()
    try:
        res, prof = profiled(e, lambda: _products_call(e, X, sj))
        counts = kernel_counts(prof, r"^(BatchProductsBody|PowerBody)<")
        assert counts == {("BatchProductsBody",): 6}, counts
        res2 = _products_call(e, X, sj)
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(res[2:], res2[2:]))
        _, prof = profiled(e, lambda: e.cwt_batch(X, 1.0, sj, _engine.MORLET, 6.0, _engine.F32))
        counts = kernel_counts(prof, r"^(BatchProductsBody|PowerBody)<")
        assert counts == {("PowerBody",): 6}, counts
    finally:
        e.close()
