"""CPU side of the row-selection / preprocessing kernel tests (no GPU).

The GPU file compares the kernels with tests/rowsel_preprocess_reference.py.  Here that reference is itself pinned:
the rolling statistic bit for bit to `sglm_pp.detrend_data(..., device=False)` (pandas' rolling apply of
`lambda_min_max`), the gather and the lag-row validity to the C oracle's gather.  The argument checks of the
entry points are exercised too: every call below fails before any CUDA call, so no device is needed."""
import ctypes

import numpy as np
import pandas as pd
import pytest

import _sglm_native as nat
import rowsel_preprocess_reference as ref
import sglm_pp
from oracle import sglm_oracle as orc

E_INVALID, E_SHAPE, E_ALIGN, E_WORKSPACE = -1, -2, -3, -4


def _same(a, b):
    """Bit-equal, except that every NaN equals every NaN."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))))


def _series(kind, n, rng):
    if kind == "walk":
        return np.cumsum(rng.standard_normal(n))
    if kind == "events":                                    # 0/1: ties everywhere, constant windows
        return (rng.random(n) < 0.15).astype(np.float64)
    x = np.cumsum(rng.standard_normal(n))
    if kind == "nan":
        x[rng.choice(n, 6, replace=False)] = np.nan
        x[0] = np.nan
    elif kind == "inf":
        x[rng.choice(n, 4, replace=False)] = np.inf
        x[rng.choice(n, 4, replace=False)] = -np.inf
    return x


@pytest.mark.parametrize("W", [2, 3, 20, 21, 40, 64])
@pytest.mark.parametrize("kind", ["walk", "events", "nan", "inf"])
def test_rolling_reference_equals_pandas(W, kind):
    rng = np.random.default_rng(1000 * W + len(kind))
    x = _series(kind, 400, rng)
    want = pd.Series(x).rolling(W, center=True).apply(sglm_pp.lambda_min_max).to_numpy()
    got = ref.rolling_minmax(x, W)
    assert _same(got, want)
    if W % 2 == 0:                                          # detrend_data takes the half window
        df = pd.DataFrame({"v": x})
        assert _same(got, sglm_pp.detrend_data(df, "v", [], W // 2, device=False).to_numpy())


@pytest.mark.parametrize("W", [4, 20])
def test_rolling_reference_grouped_equals_detrend_data(W):
    """Groups shorter than the window, one of exactly W rows, interleaved rows of several groups: pandas orders the
    result by group key, rows of a group in their original order."""
    rng = np.random.default_rng(W)
    sizes = {3: W - 1, 1: W, 0: 150, 2: 90, 4: 1}
    g = np.concatenate([np.full(s, k) for k, s in sizes.items()])
    rng.shuffle(g)
    x = np.cumsum(rng.standard_normal(len(g)))
    x[rng.choice(len(g), 3, replace=False)] = np.nan
    df = pd.DataFrame({"v": x, "g": g})
    want = sglm_pp.detrend_data(df, "v", ["g"], W // 2, device=False)
    order = np.concatenate([np.flatnonzero(g == k) for k in sorted(sizes)])
    lo, hi = ref.segments_of([sizes[k] for k in sorted(sizes)])
    got = ref.rolling_minmax(x[order], W, lo, hi)
    assert _same(got, want.to_numpy())
    assert np.array_equal(want.index.get_level_values(1).to_numpy(), order)


def _lag_cases():
    shifts_mixed = [0, 1, -1, 3, -4, 7]
    return [("mixed", [0, 1, 2, 0, 2, 1], shifts_mixed), ("positive", [2, 0, 1], [1, 5, 2]),
            ("negative", [1, 1, 0], [-2, -6, -1]), ("beyond T", [0, 1], [40, -3]), ("none", [], [])]


@pytest.mark.parametrize("case", _lag_cases(), ids=lambda c: c[0])
@pytest.mark.parametrize("fill", [np.nan, 0.0, -7.5])
def test_lag_reference_equals_oracle_gather(case, fill):
    """gather is the oracle's; lag_valid is `~isnan(gather).any(1)` for a NaN fill and ignores the fill otherwise
    (only NaN of the base signals count), also for a NaN in a base column no design column reads (column 3)."""
    _, src, sh = case
    rng = np.random.default_rng(len(src))
    T = 30
    X = rng.standard_normal((T, 4))
    X[[0, T - 1, 11], [0, 1, 2]] = np.nan
    X[5, 3] = np.nan
    want = orc.timeshift_c(X, np.array(src, np.int32), np.array(sh, np.int32), fill)
    got = ref.gather(X, src, sh, fill)
    assert _same(got, want)
    valid = ref.lag_valid(X, src, sh, bool(np.isnan(fill)))
    base_only = ~np.isnan(orc.timeshift_c(X, np.array(src, np.int32), np.array(sh, np.int32), 0.0)).any(axis=1)
    assert np.array_equal(valid, ~np.isnan(want).any(axis=1) if np.isnan(fill) else base_only)
    X3 = X.copy()
    X3[5, 3] = 0.0                                          # column 3 is read by no design column
    assert np.array_equal(valid, ref.lag_valid(X3, src, sh, bool(np.isnan(fill))))
    s = ref.lag_summary(valid)
    assert s[0] == valid.sum() and (s[0] == 0 or (valid[s[1]] and valid[s[2]]))


def test_row_set_references():
    idx = np.array([5, 2, 9, -1, 10, 2, 7])
    m, dup = ref.index_mask(idx, 10)
    assert np.array_equal(np.flatnonzero(m), [2, 5, 7, 9]) and dup
    assert not ref.index_mask([3, 1, -4, 12, 12], 10)[1]               # out-of-range repeats never count
    assert np.array_equal(ref.compact(np.array([0, 3, 0, 255, 1], np.uint8)), [1, 3, 4])
    assert np.array_equal(ref.compact(np.array([0, 3, 0, 255, 3], np.uint8), 3), [1, 4])
    sig = ref.signatures([[0, 2], [2, 3, 99]], 4, bits=[0, 62])
    assert sig.tolist() == [1, 0, 1 | (1 << 62), 1 << 62]


# --------------------------------------------------------------------------- argument checks (no CUDA call)
P = ctypes.c_void_p(4096)                    # aligned, never dereferenced


def test_rolling_minmax_args():
    lib = nat.lib()
    for W in (1, 16385, 0, -3):
        assert lib.sglm_rolling_minmax_f64(P, 100, None, None, W, P, None) == E_SHAPE
    assert b"window" in lib.sglm_last_error()
    assert lib.sglm_rolling_minmax_f64(P, 100, P, None, 20, P, None) == E_INVALID
    assert lib.sglm_rolling_minmax_f64(P, 100, None, P, 20, P, None) == E_INVALID
    assert lib.sglm_rolling_minmax_f64(P, -1, None, None, 20, P, None) == E_SHAPE


def test_roll_rejects_aliasing():
    lib = nat.lib()
    assert lib.sglm_roll_f64(P, 10, 3, P, None) == E_INVALID
    assert lib.sglm_roll_f64(P, -1, 3, ctypes.c_void_p(8192), None) == E_SHAPE


def test_match_compact_rejects_non_byte_match():
    lib = nat.lib()
    for match in (-1, 256, 1 << 20):
        assert lib.sglm_match_compact_rows(P, 100, match, P, P, 1 << 20, None) == E_INVALID


def test_index_mask_rejects_misaligned_mask():
    lib = nat.lib()
    for off in (1, 2, 3):
        assert lib.sglm_index_mask_u8(P, 10, ctypes.c_void_p(4096 + off), 100, P, None) == E_ALIGN
    assert lib.sglm_index_mask_u8(P, -1, P, 100, P, None) == E_SHAPE
    assert lib.sglm_index_mask_u8(None, 10, P, 100, P, None) == E_INVALID


def test_rows_or_bit_rejects_bit_63():
    lib = nat.lib()
    for bit in (63, 64, -1):
        assert lib.sglm_rows_or_bit_u64(P, 10, bit, P, 100, None) == E_SHAPE


@pytest.mark.parametrize("T", [1, 4096, 4097, 1024 * 4096 + 1])
def test_mask_compact_workspace(T):
    lib = nat.lib()
    need = lib.sglm_mask_compact_workspace_bytes(T)
    assert need == -(-T // 4096) * 8
    assert lib.sglm_mask_compact_rows(P, T, P, P, need - 8, None) == E_WORKSPACE
    assert lib.sglm_match_compact_rows(P, T, 0, P, P, need - 1, None) == E_WORKSPACE


@pytest.mark.parametrize("T,C", [(1, 1), (4096, 256), (4097, 257), (3 * 4096 + 5, 600)])
def test_col_moments_workspace(T, C):
    lib = nat.lib()
    need = lib.sglm_col_moments_workspace_bytes(T, C)
    assert need == (2 * -(-T // 4096) + 1) * C * 8
    assert lib.sglm_col_moments_f64(P, C, T, C, 0, 0, P, P, P, need - 1, None) == E_WORKSPACE
    assert lib.sglm_col_moments_f64(P, C - 1, T, C, 0, 0, P, P, P, need, None) == E_SHAPE
