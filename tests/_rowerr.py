"""Row-relative error measure for transforms whose rows are computed one by one.

The parity metric of the suite (conftest.relerr) divides by the largest coefficient of the
whole transform, so a row that is 1e-4 of that maximum may be wrong in its fourth digit and
still pass.  Rows of W are produced independently (each scale has its own plan: pruned
transform, dense transform or coarse transform + expansion), so they are measured one by one:

    max|W_j - Wr_j| <= tol_row * max|Wr_j| + tol_abs * max|Wr|

The second term covers rows that are tiny by construction (scales below Nyquist or far
beyond the record), where the band cut-off of the engine (1e-16 of the response peak) is not
small relative to the row itself.  Use white-noise inputs: a flat spectrum does not amplify
the rounding of the shared forward FFT for any row, so the row-relative gate is meaningful."""
import numpy as np


def row_errors(W, Wr):
    """(max|W_j - Wr_j|, max|Wr_j|) per row, and max|Wr|."""
    W = np.asarray(W)
    Wr = np.asarray(Wr)
    assert W.shape == Wr.shape, (W.shape, Wr.shape)
    assert np.isfinite(W).all() and np.isfinite(Wr).all()
    W2, Wr2 = W.reshape(-1, W.shape[-1]), Wr.reshape(-1, Wr.shape[-1])
    d = np.abs(W2 - Wr2).max(axis=1)
    r = np.abs(Wr2).max(axis=1)
    return d, r, float(r.max()) if r.size else 0.0


def check_rows(W, Wr, tol_row, tol_abs, what=""):
    """Assert the row gate above for every row of W [rows, n] (or [..., rows, n]).  Returns
    the worst row-relative error max_j max|W_j - Wr_j| / max|Wr_j| over the rows the first
    term governs (max|Wr_j| >= tol_abs / tol_row * max|Wr|)."""
    d, r, g = row_errors(W, Wr)
    bound = tol_row * r + tol_abs * g
    bad = np.nonzero(d > bound)[0]
    assert bad.size == 0, "%s: rows %s exceed the row gate: err %s, row max %s, max|Wr| %.3e" % (
        what, bad[:8].tolist(), d[bad[:8]].tolist(), r[bad[:8]].tolist(), g)
    big = r >= (tol_abs / tol_row) * g
    return float((d[big] / r[big]).max()) if big.any() else 0.0
