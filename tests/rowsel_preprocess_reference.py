"""Plain numpy definitions of the row-selection kernels (csrc/timeshift.cu) and the preprocessing kernels
(csrc/preprocess.cu): what each entry point must compute, written the obvious way.  A helper of
tests/test_rowsel_preprocess_cpu.py and tests/test_gpu_rowsel_preprocess.py, not a test module itself.

  gather            out[t, c] = X[t - shift_c, src_c], or `fill` where t - shift_c falls outside [0, T)
  lag_valid         rows of the gathered design without NaN; with a non-NaN fill only the base signals' NaNs count
  compact           np.flatnonzero of a byte mask (any non-zero byte is set), or of `ids == match`
  index_mask        np.bincount of the in-range positions of an index list: (row mask, some row listed twice)
  signatures        bit b of sig[t] set when row t is listed in set b
  col_moments       column mean and sd in longdouble; numpy's rules (ddof 0, NaN propagates) or pandas'
                    (ddof 1, NaN skipped; sd NaN when at most ddof values remain)
  rolling_minmax    pandas' `rolling(W, center=True).apply(lambda_min_max)`: the W-window ending (W - 1) // 2 rows
                    right of the labelled row, np.quantile(window, [0.05, 0.95]) (linear), then
                    (centre - q05) / (q95 - q05) with centre = window[(W + 1) // 2 - 1]; NaN unless the window lies
                    inside its segment and holds only finite values (pandas' rolling turns +-inf into NaN before
                    it counts the observations of a window)"""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view

LD = np.longdouble
_ROLL_CHUNK_ELEMS = 1 << 22          # window values handed to one np.quantile call


def gather(X, src, shift, fill):
    """Moves bits, never values: a NaN fill keeps its payload, -0.0 its sign."""
    Xb = np.ascontiguousarray(X, dtype=np.float64).view(np.uint64)
    T = Xb.shape[0]
    src = np.asarray(src, dtype=np.int64)
    shift = np.asarray(shift, dtype=np.int64)
    out = np.full((T, len(src)), np.array(fill, dtype=np.float64).view(np.uint64), dtype=np.uint64)
    t = np.arange(T)
    for c, (p, s) in enumerate(zip(src, shift)):
        ts = t - s
        ok = (ts >= 0) & (ts < T)
        out[ok, c] = Xb[ts[ok], p]
    return out.view(np.float64)


def lag_valid(X, src, shift, fill_is_nan):
    """Rows of gather(X, src, shift, fill) without NaN, for a NaN fill or (fill_is_nan False) any non-NaN fill."""
    return ~np.isnan(gather(X, src, shift, np.nan if fill_is_nan else 0.0)).any(axis=1)


def lag_summary(valid):
    """{count, first set row, last set row}; {0, T, -1} when no row is set."""
    nz = np.flatnonzero(valid)
    return np.array([nz.size, nz[0] if nz.size else len(valid), nz[-1] if nz.size else -1], dtype=np.int64)


def compact(mask, match=None):
    mask = np.asarray(mask)
    return np.flatnonzero(mask != 0 if match is None else mask == match).astype(np.int64)


def index_mask(idx, T):
    """(uint8 mask of the rows listed in [0, T), whether an in-range row is listed more than once)."""
    idx = np.asarray(idx, dtype=np.int64)
    n = np.bincount(idx[(idx >= 0) & (idx < T)], minlength=T)
    return (n > 0).astype(np.uint8), bool((n > 1).any())


def signatures(sets, T, bits=None):
    sig = np.zeros(T, dtype=np.uint64)
    for k, rows in enumerate(sets):
        b = k if bits is None else bits[k]
        rows = np.asarray(rows, dtype=np.int64)
        sig[rows[(rows >= 0) & (rows < T)]] |= np.uint64(1) << np.uint64(b)
    return sig


def col_moments(X, ddof, skipna):
    """Longdouble (mean, sd, n, sum |x|) per column, NaN entries skipped (skipna) or propagated."""
    X = np.asarray(X, dtype=np.float64)
    nan = np.isnan(X)
    Xl = X.astype(LD)
    if skipna:
        Xl = np.where(nan, LD(0), Xl)
        n = (~nan).sum(axis=0)
    else:
        n = np.full(X.shape[1], X.shape[0])
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = Xl.sum(axis=0) / n
        d = Xl - mean
        if skipna:
            d = np.where(nan, LD(0), d)
        var = (d * d).sum(axis=0) / (n - ddof)
        sd = np.where(n > ddof, np.sqrt(var), LD(np.nan))
        if not skipna:
            sd = np.where(nan.any(axis=0), LD(np.nan), sd)
    return mean, sd, n, np.abs(Xl).sum(axis=0)


def zscore(X, mean, sd):
    return (X - mean) / sd


def _rolling_segment(x, W):
    n = len(x)
    out = np.full(n, np.nan)
    if n < W:
        return out
    off_r = (W - 1) // 2
    m = n - W + 1                                  # windows x[j: j + W], j < m, labelled at j + W - 1 - off_r
    step = max(1, _ROLL_CHUNK_ELEMS // W)
    win_all = sliding_window_view(x, W)
    for j0 in range(0, m, step):
        win = win_all[j0: j0 + step]
        centre = win[:, (W + 1) // 2 - 1]
        with np.errstate(all="ignore"):
            q = np.quantile(win, [0.05, 0.95], axis=1)
            v = (centre - q[0]) / (q[1] - q[0])
        v[~np.isfinite(win).all(axis=1)] = np.nan
        out[j0 + W - 1 - off_r: j0 + W - 1 - off_r + len(v)] = v
    return out


def rolling_minmax(x, W, seg_lo=None, seg_hi=None):
    """The rolling statistic of every row of x; seg_lo / seg_hi: per-row bounds [lo, hi) of contiguous segments."""
    x = np.asarray(x, dtype=np.float64)
    if seg_lo is None:
        return _rolling_segment(x, W)
    out = np.full(len(x), np.nan)
    for lo, hi in sorted(set(zip(np.asarray(seg_lo).tolist(), np.asarray(seg_hi).tolist()))):
        out[lo:hi] = _rolling_segment(x[lo:hi], W)
    return out


def segments_of(sizes):
    """Per-row [seg_lo, seg_hi) of consecutive segments of the given sizes."""
    sizes = np.asarray(sizes, dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    return np.repeat(starts[:-1], sizes), np.repeat(starts[1:], sizes)
