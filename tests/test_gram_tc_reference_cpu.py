"""CPU side of the tensor-core Gram tests (no GPU).

tests/test_gpu_gram_stats_kernels.py compares the kernels of csrc/gram_tc.cu bit for bit with the model in
tests/gram_tc_reference.py.  Here the model itself is pinned: its plane counts against the digit-by-digit expansion,
its digits against the values they represent, its Gram against the exact Gram of those values (Python fractions),
and its plan against the layout rules of tc_make_plan.  The argument checks of the entry points run too: every call
below fails on the host before any CUDA call, so no device is needed."""
import ctypes
from fractions import Fraction

import numpy as np
import pytest

import _sglm_native as nat
import gram_tc_reference as ref

E_INVALID, E_SHAPE, E_UNSUPPORTED = -1, -2, -6


def _catalogue_Z(T=300, seed=1):
    rng = np.random.default_rng(seed)
    cols = ref.catalogue(T, rng)
    return list(cols), np.stack(list(cols.values()), axis=1)


def _exact(x):
    return Fraction(float(x))


def test_plane_count_equals_digit_expansion():
    """The lowest-set-bit count (tc_exponent_kernel) equals the largest digit-by-digit count (tc_digits_kernel) of the
    column's values: no value needs more planes than the column gets, and the column gets no plane none of its
    values needs.  Uncapped, the count is >= 8 exactly when the expansion does not end within 8 planes."""
    names, Z = _catalogue_Z()
    a = ref.analyze(Z)
    uncapped = ref.exponents(a["colmax_bits"], a["col_lsb"], max_planes=99)[1]
    for c, name in enumerate(names):
        E = int(a["colE"][c])
        need = max([1] + [ref.digits_needed(z, E) for z in Z[:, c]])
        assert int(a["colS"][c]) == need, name
        assert (need == 8) == (uncapped[c] >= 8), name


def test_analysis_of_special_columns():
    names, Z = _catalogue_Z()
    a = ref.analyze(Z)
    col = dict(zip(names, range(len(names))))
    assert a["colE"][col["all_zero"]] == 0 and a["colS"][col["all_zero"]] == 1
    assert a["col_lsb"][col["all_zero"]] == ref.EMPTY_LSB
    assert a["colE"][col["pow2_pos"]] == 11                      # 2^10 < 2^11
    assert a["colE"][col["pow2_neg_max"]] == -2
    assert a["colS"][col["zero_one"]] == 1 and a["colS"][col["constant"]] == 1
    assert a["colS"][col["one_plus_tiny"]] == 8 and a["colS"][col["one_plus_ulp"]] == 8
    assert a["col_lsb"][col["subnormal_mix"]] == -1074
    for e in (899, 900, 901, -899, -900, -901):
        assert a["colE"][col[f"e{e}"]] == e
    for m in (1, 4, 8):
        assert np.array_equal(ref.analyze(Z, max_planes=m)["colS"], np.minimum(a["colS"], m))
    bad = Z.copy()
    bad[3, 2] = np.nan
    bad[5, 4] = np.inf
    b = ref.analyze(bad)
    assert b["flag"] == 1 and b["colmax_bits"][2] == ref.NAN_BITS and b["colmax_bits"][4] == ref.NAN_BITS
    assert b["colE"][2] == 0 and b["colS"][2] == 1
    empty = ref.analyze(Z[:0])
    assert empty["flag"] == 0 and not empty["colmax_bits"].any() and np.all(empty["colS"] == 1)


@pytest.mark.parametrize("max_planes", [1, 2, 4, 8])
def test_digits_reconstruct_values(max_planes):
    """sum_k d_k 2^(E - 6 - 7(k - 1)) == z exactly when the column needs at most S planes, else within 2^(E - 7S)
    (half a unit of the last kept plane).  Every digit lies in [-64, 64]."""
    names, Z = _catalogue_Z()
    a = ref.analyze(Z, max_planes=max_planes)
    uncapped = ref.exponents(a["colmax_bits"], a["col_lsb"], 99)[1]
    planes = ref.digits(Z, None, a["colE"], a["colS"])
    worst = {}
    for c, name in enumerate(names):
        E, S = int(a["colE"][c]), int(a["colS"][c])
        d = planes[c].astype(np.int64)
        assert np.abs(d).max() <= 64, name
        for t in range(0, Z.shape[0], 3):
            rec = sum(Fraction(int(d[k, t])) * Fraction(2) ** (E - 6 - 7 * k) for k in range(S))
            err = abs(rec - _exact(Z[t, c]))
            if uncapped[c] <= S:
                assert err == 0, (name, t)
            else:
                assert err <= Fraction(2) ** (E - 7 * S), (name, t)
            worst[name] = max(worst.get(name, 0), err / Fraction(2) ** (E - 7 * S))
    if max_planes == 1:
        assert worst["ties"] == 1          # a tie at the last kept plane reaches the bound: it is 2^(E - 7S), not less


def _exact_gram(planes, colE, colS, rows):
    """Exact Gram (fractions) of the values the digits represent."""
    n = len(planes)
    vals = []
    for c in range(n):
        w = [Fraction(2) ** (int(colE[c]) - 6 - 7 * k) for k in range(int(colS[c]))]
        vals.append([sum(int(planes[c][k, t]) * w[k] for k in range(int(colS[c]))) for t in rows])
    return [[sum(vals[i][r] * vals[j][r] for r in range(len(rows))) for j in range(n)] for i in range(n)]


def test_gram_against_fractions():
    """gram() against the exact Gram of the represented values.  Its error comes from the dropped k + l > 9 pairs
    (each |d d'| <= 2^12 per row at weight 2^(E1 + E2 - 12 - 7(tot - 2)), tot >= 10) and the eight `acc +=`
    roundings plus the final scaling (at most 9 u |acc|, with |acc| bounded by the sum of |term| over the kept pairs),
    plus half the smallest subnormal when the final scaling underflows (the column near 2^-899)."""
    rng = np.random.default_rng(5)
    T = 64
    cols = ref.catalogue(T, rng)
    keep = ["gauss", "ties", "one_plus_ulp", "one_plus_tiny", "first_digit_64", "dyadic", "pow2_neg_max", "e-899"]
    Z = np.stack([cols[k] for k in keep] + [np.ones(T)], axis=1)
    rows = np.sort(rng.choice(T, 40, replace=False))
    G, a = ref.gram(Z, [rows])
    E, S = a["colE"], a["colS"]
    planes = ref.digits(Z, None, E, S)
    exact = _exact_gram(planes, E, S, rows)
    n = Z.shape[1]
    for i in range(n):
        for j in range(n):
            mag = Fraction(0)
            dropped = Fraction(0)
            for k in range(1, int(S[i]) + 1):
                for l in range(1, int(S[j]) + 1):
                    s = sum(abs(int(planes[i][k - 1, t]) * int(planes[j][l - 1, t])) for t in rows)
                    w = Fraction(2) ** (int(E[i]) + int(E[j]) - 12 - 7 * (k + l - 2))
                    if k + l > 9:
                        dropped += s * w
                    else:
                        mag += s * w
            bound = dropped + 9 * Fraction(2) ** -53 * mag + Fraction(2) ** -1075   # + underflow of the final scaling
            assert abs(_exact(G[0, i, j]) - exact[i][j]) <= bound, (keep[i] if i < len(keep) else "1",
                                                                    keep[j] if j < len(keep) else "1")
    assert np.array_equal(G[0].view(np.uint64), G[0].T.view(np.uint64))


def test_gram_exact_for_short_columns():
    """Integer, 0/1 and dyadic columns with S1 + S2 <= 9: every plane pair is kept and every partial sum is exact, so
    gram() is Z'Z exactly."""
    rng = np.random.default_rng(7)
    T = 500
    Z = np.stack([(rng.random(T) < 0.3).astype(np.float64), rng.integers(-50, 50, T).astype(np.float64),
                  rng.integers(-2 ** 12, 2 ** 12, T) * 2.0 ** -7, rng.integers(0, 3, T).astype(np.float64),
                  np.ones(T)], axis=1)
    sets = [np.arange(T), np.arange(0, T, 3), np.array([], dtype=np.int64), np.array([17])]
    G, a = ref.gram(Z, sets)
    S = a["colS"]
    assert (S[:, None] + S[None, :]).max() <= 9
    for g, rows in zip(G, sets):
        want = Z[rows].T @ Z[rows]                  # exact: integers / dyadics far below 2^53
        assert np.array_equal(g, want)


@pytest.mark.parametrize("n_aug", [255, 256, 257, 513])
def test_plan_layout(n_aug):
    rng = np.random.default_rng(n_aug)
    colS = rng.choice([1, 1, 1, 2, 3, 8], n_aug)
    colS[-1] = 1
    p = ref.plan(n_aug, colS, [1000, 0, 129, 2048 * 128 + 1])
    assert p["S"] % 256 == 0 and p["level_cnt"][1] == n_aug
    for (mt, nt), (k, l) in zip(p["tiles"], p["tile_levels"]):
        assert k <= l and k + l <= 9
        if k == l:
            assert (nt + 1) * ref.TC_BN > mt * ref.TC_BM          # not strictly below the diagonal
    for c in range(n_aug):
        rows = p["plane_row"][c]
        assert np.all(rows[:colS[c]] >= 0) and np.all(rows[colS[c]:] == -1)
    used = p["plane_row"][p["plane_row"] >= 0]
    assert len(np.unique(used)) == len(used) == colS.sum()
    # the set of 262145 rows is cut into K segments of at most 2048 blocks of 128 rows
    assert [s[1] for s in p["segs"] if s[2] == 3] == [2048, 1]
    assert [s[1] for s in p["segs"] if s[2] == 1] == [0]


# --------------------------------------------------------------------------- argument checks (host only)
def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _rc(name, *args):
    return getattr(nat.lib(), name)(*args)


@pytest.mark.parametrize("max_planes", [0, 9, -1])
def test_max_planes_refused(max_planes):
    buf = np.zeros(64)
    assert _rc("sglm_gram_tc_analyze_scaled_f64", _p(buf), 1, None, 0, 0, 4, 1, _p(buf), max_planes, _p(buf), _p(buf),
               _p(buf), _p(buf), None) == E_INVALID
    assert _rc("sglm_gram_tc_exponents", _p(buf), 2, max_planes, _p(buf), _p(buf), _p(buf), None) == E_INVALID


def test_null_pointers_refused():
    buf = np.zeros(64)
    i32 = np.ones(4, dtype=np.int32)
    rows = np.full(4, 128, dtype=np.int64)
    assert _rc("sglm_gram_tc_analyze_f64", _p(buf), 1, None, 0, 0, 4, 1, None, _p(buf), _p(buf), _p(buf), None) == E_INVALID
    assert _rc("sglm_gram_tc_colstats_f64", _p(buf), 1, None, 0, 0, 4, 1, None, _p(buf), None) == E_INVALID
    assert _rc("sglm_gram_tc_colstats_scaled_f64", _p(buf), 1, None, 0, 0, 4, 1, None, _p(buf), _p(buf), None) == E_INVALID
    assert _rc("sglm_gram_tc_exponents", None, 2, 8, _p(buf), _p(buf), _p(buf), None) == E_INVALID
    assert _rc("sglm_gram_tc_plan_info", 2, None, 1, _p(rows), _p(rows)) == E_INVALID
    assert _rc("sglm_gram_tc_f64", _p(buf), 1, None, 0, 0, 4, 1, None, _p(i32), _p(i32), 1, _p(rows), _p(rows), _p(buf),
               2, _p(buf), 1 << 20, 0, None) == E_INVALID
    assert _rc("sglm_gram_tc_f64", _p(buf), 1, None, 0, 0, 4, 1, _p(i32), _p(i32), _p(i32), 1, _p(rows), _p(rows), _p(buf),
               1, _p(buf), 1 << 20, 0, None) == E_SHAPE                    # ldg < n_aug
    assert _rc("sglm_gram_tc_cells_f64", _p(buf), 1, None, 0, 0, 4, 1, _p(i32), _p(i32), _p(i32), 1, _p(rows), _p(rows), 1,
               None, _p(buf), 2, _p(buf), 1 << 20, 0, None) == E_INVALID   # membership table missing
    assert _rc("sglm_gram_tc_cells_f64", _p(buf), 1, None, 0, 0, 4, 1, _p(i32), _p(i32), _p(i32), 257, _p(rows), _p(rows), 1,
               _p(i32), _p(buf), 2, _p(buf), 1 << 20, 0, None) == E_UNSUPPORTED
    assert _rc("sglm_gram_tc_scaled_partial_f64", _p(buf), 1, None, 0, 0, 4, 1, None, _p(i32), _p(i32), _p(i32), 1,
               _p(rows), _p(rows), 1, _p(i32), _p(buf), 1 << 20, None) == E_INVALID      # row_scale missing, T > 0
    assert _rc("sglm_gram_tc_lag_cells_f64", None, None, 0, 0, 4, 1, _p(i32), _p(i32), _p(i32), 1, _p(rows), _p(rows), 0,
               None, _p(buf), 2, _p(buf), 1 << 20, 0, None) == E_INVALID
    lag = nat.LagDesignStruct(0, 1, 4, 1, 0, 0, 0, 0, 0)
    assert _rc("sglm_gram_tc_lag_cells_f64", ctypes.byref(lag), None, 0, 0, 4, 1, _p(i32), _p(i32), _p(i32), 1, _p(rows),
               _p(rows), 0, None, _p(buf), 2, _p(buf), 1 << 20, 1, None) == E_INVALID  # partial without output sets
    assert _rc("sglm_center_stats_f64", None, None, 4, 1, 1, 0, 1, _p(buf), 1, _p(buf), _p(buf), _p(buf), _p(buf),
               None) == E_INVALID
    assert _rc("sglm_center_stats_f64", _p(buf), None, 2, 1, 1, 0, 1, _p(buf), 1, _p(buf), _p(buf), _p(buf), _p(buf),
               None) == E_SHAPE                                            # ldg < C + n_y + 1
    assert _rc("sglm_finalize_models_f64", _p(buf), 2, 2, 1, None, None, None, 1, None, None, 0, None) == E_INVALID
    assert _rc("sglm_finalize_models_f64", _p(buf), 2, 2, 1, None, _p(buf), None, 1, _p(buf), None, 0, None) == E_INVALID
    assert _rc("sglm_finalize_models_f64", _p(buf), 2, 2, 1, None, None, None, 1, _p(buf), _p(buf), 3, None) == E_SHAPE
    assert _rc("sglm_quadform_f64", None, 4, 4, _p(buf), 4, 1, _p(buf), None) == E_INVALID
    assert _rc("sglm_quadform_gemm_f64", _p(buf), 4, 4, None, 64, 1, _p(buf), _p(buf), _p(buf), None) == E_INVALID
    assert _rc("sglm_quadform_gemm_f64", _p(buf), 4, 4, _p(buf), 32, 1, _p(buf), _p(buf), _p(buf), None) == E_SHAPE
    assert _rc("sglm_index_counts_f64", None, 3, _p(buf), 4, None) == E_INVALID
    ks = np.ones(2, dtype=np.int32)
    assert _rc("sglm_suffstats_f64", _p(buf), 1, _p(buf), 1, 1, 4, 1, None, 0, 1, _p(ks), None, 3, _p(buf), 1 << 20,
               None) == E_INVALID
    assert _rc("sglm_suffstats_f64", _p(buf), 1, _p(buf), 1, 1, 4, 1, None, 0, 0, _p(ks), _p(buf), 3, _p(buf), 1 << 20,
               None) == E_SHAPE


@pytest.mark.parametrize("n_splits", [0, 65536])
def test_quadform_split_count_refused(n_splits):
    buf = np.zeros(64)
    assert _rc("sglm_quadform_split_f64", _p(buf), 4, 4, _p(buf), 4, 1, n_splits, _p(buf), None) == E_INVALID


def test_quadform_too_large_for_shared_memory():
    """n = 7265: the 4-model form needs 4 n 8 bytes > 227 KB of shared memory; refused before any launch (the buffers
    are host memory the call never touches)."""
    buf = np.zeros(64)
    n = 227 * 1024 // 32 + 1
    assert _rc("sglm_quadform_f64", _p(buf), n, n, _p(buf), n, 3, _p(buf), None) == E_UNSUPPORTED
    assert _rc("sglm_quadform_split_f64", _p(buf), n, n, _p(buf), n, 3, 4, _p(buf), None) == E_UNSUPPORTED
