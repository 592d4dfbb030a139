"""Kernel-level references for the row-selection kernels (csrc/timeshift.cu) and the preprocessing kernels
(csrc/preprocess.cu).  Every entry point is called directly and compared with tests/rowsel_preprocess_reference.py.

Exact results are required everywhere except the column moments:
  - row lists, masks, flags, signatures, cell tables, gathers, rolls and crops move or count bits: equal bits;
  - z-scores and first differences are one IEEE operation per element: equal to numpy's bits (NaN positions only
    where the result is NaN, since NaN payloads are platform-defined);
  - the rolling statistic sorts exactly, interpolates as numpy's _lerp does (product rounded, then the sum) and
    divides once: equal to the reference (pandas), with +-0.0 equal and NaN positions matching.
Output buffers are longer than the result and pre-filled with a sentinel that must survive, so a kernel that writes
one element too many fails.

Column moments (sglm_col_moments_f64): the sum over t runs sequentially inside a chunk of L = min(T, 4096) rows and
then sequentially over the K = ceil(T / 4096) chunk partials.  Recursive summation of terms x_i has
|err| <= gamma_(k-1) sum |x_i| (gamma_k = k u / (1 - k u), u = 2^-53); the two levels compose to
gamma_(L+K-2) sum |x|, and the division by n adds u |mean|.  With gamma_k <= 1.01 k u (k u < 0.01 here):
    |mean_gpu - mean| <= 2 (L + K) u sum|x| / n.                                                           (1)
The second pass sums d_t^2, d_t = fl(x_t - m) with the device mean m; each term carries at most 3 roundings (the
difference, the square, the addition; fewer when contracted), so with Q(m) = sum (x_t - m)^2
    |Q_gpu - Q(m)| <= 2 (L + K + 3) u Q(m),   Q(m) = Q(mean) + n (m - mean)^2   (exact: sum (x - mean) = 0),
and var = Q / (n - ddof) adds one rounding:
    bv = [2 (L + K + 4) u Q(m) + n (m - mean)^2] / (n - ddof)                                              (2)
bounds |var_gpu - var|, with (m - mean) the measured error of the device mean.  The square root then gives
    |sd_gpu - sd| <= min(sqrt(bv), bv / sd) + 2 u (sd + sqrt(bv))                                          (3)
(|sqrt(a) - sqrt(b)| <= min(sqrt|a - b|, |a - b| / sqrt(b)); the rounded sqrt adds u sd_gpu, and
sd_gpu <= (sd + sqrt(bv)) (1 + u)).  The reference is numpy longdouble (64-bit mantissa): its own error is 2^-11
of these bounds and is not added.  A one-pass formula sum x^2 / n - mean^2 cannot resolve the variance of a
1e8 + N(0, 1) column at all: both terms lie near 1e16, where doubles are 2 apart."""
import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import _engine as eng  # noqa: E402
import _sglm_native as nat  # noqa: E402
import rowsel_preprocess_reference as ref  # noqa: E402
import sglm_pp  # noqa: E402
from oracle import sglm_oracle as orc  # noqa: E402

LD = np.longdouble
U = 2.0 ** -53
F64 = torch.float64
I64 = torch.int64
SENT = -0x5A5A5A5A5A5A5A5B                  # int64 sentinel of the tails
SENT_F = np.array([SENT], dtype=np.int64).view(np.float64)[0]          # the same bits as a (NaN) double
CH = 4096                                   # rows per block of the ordered compaction / per chunk of the moments


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(device="cuda", dtype=dtype) if dtype is not None else t.to("cuda")


def _st():
    return nat.stream_ptr()


def _host(t):
    return t.detach().cpu().numpy()


def _bits(a):
    a = np.ascontiguousarray(_host(a) if torch.is_tensor(a) else a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def _same_bits(got, want, what):
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    bad = np.flatnonzero((g != w).reshape(-1))
    assert bad.size == 0, f"{what}: {bad.size} of {g.size} differ; first at {bad[0]}: {g.reshape(-1)[bad[0]]:#x} vs " \
                          f"{w.reshape(-1)[bad[0]]:#x}"


def _same_values(got, want, what):
    """Equal as doubles (+0.0 == -0.0) and NaN exactly where the reference is NaN."""
    g = np.asarray(_host(got) if torch.is_tensor(got) else got, dtype=np.float64)
    w = np.asarray(want, dtype=np.float64)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    ok = (g == w) | (np.isnan(g) & np.isnan(w))
    bad = np.flatnonzero(~ok.reshape(-1))
    assert bad.size == 0, f"{what}: {bad.size} of {g.size} differ; first at {bad[0]}: got {g.reshape(-1)[bad[0]]!r}, " \
                          f"want {w.reshape(-1)[bad[0]]!r}"


def _i64_with_tail(n, tail=64):
    return torch.full((n + tail,), SENT, dtype=I64, device="cuda")


def _tail_intact(buf, n, what):
    assert bool((buf[n:] == SENT).all()), f"{what}: written past the end"


def _padded(A, ld, pad):
    """Device matrix [T][ld] holding A in its first columns and `pad` elsewhere; returns (tensor, view)."""
    T, C = A.shape
    big = torch.full((max(T, 1), ld), pad, dtype=F64, device="cuda")
    if T:
        big[:T, :C] = _dev(A)
    return big, big[:T, :C]


# --------------------------------------------------------------------------- ordered compaction
COMPACT_T = [1, 31, CH - 1, CH, CH + 1, 1024 * CH, 1024 * CH + 1, 3 * 1024 * CH + 777]


def _masks(T, rng):
    out = {"empty": np.zeros(T, np.uint8), "full": np.ones(T, np.uint8),
           "d1e-4": (rng.random(T) < 1e-4).astype(np.uint8), "d0.5": (rng.random(T) < 0.5).astype(np.uint8)}
    nb = -(-T // CH)
    blk = rng.integers(0, 3, nb)                  # whole 4096-row blocks empty (0), full (1) or half (2)
    m = np.where(np.repeat(blk, CH)[:T] == 1, 1, 0).astype(np.uint8)
    half = np.repeat(blk, CH)[:T] == 2
    m[half] = rng.random(int(half.sum())) < 0.5
    out["blocks"] = m
    b = rng.integers(0, 256, T).astype(np.uint8)
    b[rng.random(T) < 0.5] = 0                     # bytes 2..255 count as set
    out["bytes"] = b
    return out


def _compact(mask_d, T, match=None):
    count = int((mask_d[:T] != 0).sum() if match is None else (mask_d[:T] == match).sum())
    rows = _i64_with_tail(count)
    wb = nat.lib().sglm_mask_compact_workspace_bytes(T)
    ws = torch.empty((wb + 7) // 8, dtype=I64, device="cuda")
    if match is None:
        nat.call("sglm_mask_compact_rows", nat.ptr(mask_d), T, nat.ptr(rows), nat.ptr(ws), wb, _st())
    else:
        nat.call("sglm_match_compact_rows", nat.ptr(mask_d), T, match, nat.ptr(rows), nat.ptr(ws), wb, _st())
    return rows, count


@pytest.mark.parametrize("T", COMPACT_T)
def test_mask_and_match_compaction(T):
    """Ascending row indices of the set bytes, exactly `count` of them; T past 1024 blocks of 4096 rows takes the
    scan's second round (its carry).  match = 0 and 255 select by byte value."""
    rng = np.random.default_rng(T)
    for kind, m in _masks(T, rng).items():
        md = _dev(m)
        rows, count = _compact(md, T)
        _same_bits(rows[:count], ref.compact(m), f"mask_compact T={T} {kind}")
        _tail_intact(rows, count, f"mask_compact T={T} {kind}")
        if kind == "bytes":
            for match in (0, 255):
                rows, count = _compact(md, T, match)
                _same_bits(rows[:count], ref.compact(m, match), f"match_compact T={T} match={match}")
                _tail_intact(rows, count, f"match_compact T={T} match={match}")


# --------------------------------------------------------------------------- index mask, signatures, cells
@pytest.mark.parametrize("T", [4096, 4097, 4098, 4099, 1_000_003])
def test_index_mask(T):
    """mask[t] = 1 for the listed in-range rows, bytes between T and round-up-to-4(T) zeroed, bytes past that left
    alone; dup_flag = 1 exactly when an in-range row is listed twice (out-of-range repeats are ignored)."""
    rng = np.random.default_rng(T)
    r4 = (T + 3) // 4 * 4
    pick = rng.random(T) < 1 / 3
    pick[[0, T - 1]] = True
    uniq = rng.permutation(np.flatnonzero(pick))
    oor = np.array([-1, -1, T, T, T + 5, -(1 << 40)])
    cases = {"unique": uniq, "unique+out-of-range": np.concatenate([uniq, oor]),
             "repeat": np.concatenate([uniq, uniq[-1:]]), "repeat first": np.concatenate([uniq[:1], uniq]),
             "empty": np.zeros(0, np.int64), "out-of-range only": oor}
    for what, idx in cases.items():
        buf = torch.full((r4 + 16,), 0xA5, dtype=torch.uint8, device="cuda")
        flag = torch.tensor([7, SENT & 0x7FFFFFFF], dtype=torch.int32, device="cuda")
        idx_d = _dev(idx.astype(np.int64))
        nat.call("sglm_index_mask_u8", nat.ptr(idx_d), idx_d.numel(), nat.ptr(buf), T, nat.ptr(flag), _st())
        want, dup = ref.index_mask(idx, T)
        got = _host(buf)
        assert np.array_equal(got[:T], want), what
        assert not got[T:r4].any() and (got[r4:] == 0xA5).all(), what
        f = _host(flag)
        assert f[0] == int(dup) and f[1] == SENT & 0x7FFFFFFF, (what, f)


def test_rows_or_bit():
    """Bits 0 and 62; a second call with bit 0 ORs into the first; out-of-range entries are skipped."""
    T = 100_003
    rng = np.random.default_rng(3)
    lists = [rng.choice(T, 5000, replace=False), rng.choice(T, 40_000, replace=False),
             np.concatenate([rng.choice(T, 7000, replace=False), [-1, T, T + 1, -(1 << 40)]])]
    bits = [0, 62, 0]
    sig = torch.zeros(T + 8, dtype=I64, device="cuda")
    sig[T:] = SENT
    for rows, bit in zip(lists, bits):
        r = _dev(rows.astype(np.int64))
        nat.call("sglm_rows_or_bit_u64", nat.ptr(r), r.numel(), bit, nat.ptr(sig), T, _st())
    _same_bits(_host(sig[:T]).view(np.uint64), ref.signatures(lists, T, bits), "signatures")
    _tail_intact(sig, T, "signatures")


def _distinct_keys(k, rng):
    """k distinct keys below 2^63: 0, two with bit 62 set, then random ones (about half of them with bit 62)."""
    keys = [0, 1 << 62, (1 << 62) | 5]
    seen = set(keys)
    while len(keys) < k:
        v = int(rng.integers(0, 1 << 63, dtype=np.uint64))
        if v not in seen:
            seen.add(v)
            keys.append(v)
    return np.array(keys[:k], dtype=np.uint64)


def _cells(sig, table):
    T = sig.numel()
    cell_of = torch.full((T,), 0xA5, dtype=torch.uint8, device="cuda")
    nat.call("sglm_cells_from_signatures", nat.ptr(sig), T, nat.ptr(cell_of), nat.ptr(table), _st())
    th = _host(table)
    return _host(cell_of), th[:256].view(np.uint64), th[256:512], th[512:513].view(np.int32)


@pytest.mark.parametrize("k,T", [(1, 1), (1, 5000), (2, 100_000), (65, 3_000_000), (199, 300_000), (230, 300_000),
                                 (256, 300_000), (257, 300_000), (1000, 3_000_000)])
def test_cells_from_signatures(k, T):
    """k distinct signatures (key 0, keys with bit 62) over T rows.  k <= 200: no overflow, `used` = k, the keys of
    the occupied slots are the distinct signatures, their counts np.unique's, keys[cell_of[t]] = sig[t].  k > 256
    cannot fit the table: overflow.  In between either flag is right, the outputs exact whenever it is 0.  Slot
    numbers depend on atomic order, so the mapping is compared, never slot ids.  The table is reused from a call
    that overflowed: the entry point must reset it."""
    rng = np.random.default_rng(k * 7 + T)
    keys = _distinct_keys(k, rng)
    pick = rng.integers(0, k, T)
    pick[:k] = np.arange(k)[: min(k, T)]
    rng.shuffle(pick)
    sig_h = keys[pick]
    table = torch.empty(514, dtype=I64, device="cuda")
    junk = _dev(np.arange(300_000, dtype=np.uint64).view(np.int64))                   # 300k keys: overflows
    assert _cells(junk, table)[3][1] == 1
    cell_of, tkeys, counts, flags = _cells(_dev(sig_h.view(np.int64)), table)
    used, overflow = int(flags[0]), int(flags[1])
    if k <= 200:
        assert overflow == 0 and used == k, (used, overflow)
    if k > 256:
        assert overflow == 1
        return
    if overflow:
        return
    occ = np.flatnonzero(counts > 0)
    assert len(occ) == used == k
    assert (tkeys[np.setdiff1d(np.arange(256), occ)] == np.uint64(0xFFFFFFFFFFFFFFFF)).all()
    uk, uc = np.unique(sig_h, return_counts=True)
    order = np.argsort(tkeys[occ])
    assert np.array_equal(tkeys[occ][order], uk) and np.array_equal(counts[occ][order], uc)
    assert np.array_equal(tkeys[cell_of], sig_h)
    # the rows of one cell, through the byte-match compaction
    for sl in occ[:3]:
        rows, count = _compact(_dev(cell_of), T, int(sl))
        _same_bits(rows[:count], np.flatnonzero(cell_of == sl), f"match_compact cell {sl}")


def test_row_cells_overflow_falls_back_to_per_set_gram():
    """More than 200 distinct row signatures: eng._row_cells gives up (None) and the tensor-core Gram of the sets
    is the per-set pass, bit for bit."""
    T, C = 6000, 24
    rng = np.random.default_rng(11)
    sets = [None] + [torch.from_numpy(np.flatnonzero(rng.random(T) < 0.5)).cuda() for _ in range(10)]
    sig = ref.signatures([_host(s) for s in sets[1:]], T)
    assert len(np.unique(sig)) > 200
    assert eng._row_cells(sets, T) is None
    X = rng.standard_normal((T, C)).round(3)
    Xd, Yd = _dev(X), _dev(rng.standard_normal((T, 1)))
    old = eng.TC_CELLS
    try:
        eng.TC_CELLS = None
        G_auto, _ = eng.suffstats_tc(Xd, Yd, sets)
        assert not nat.last_tc_plan["cells"]
        eng.TC_CELLS = False
        G_sets, _ = eng.suffstats_tc(Xd, Yd, sets)
    finally:
        eng.TC_CELLS = old
    _same_bits(G_auto, G_sets, "suffstats_tc with too many cells")


# --------------------------------------------------------------------------- lag-row validity
def _lag_valid(Xbig, X, src, sh, fill_is_nan):
    T, P = X.shape
    valid = torch.full((max(T, 1) + 16,), 0xA5, dtype=torch.uint8, device="cuda")
    summ = torch.full((3,), SENT, dtype=I64, device="cuda")
    C = len(src)
    s_d, h_d = _dev(np.asarray(src, np.int32)), _dev(np.asarray(sh, np.int32))
    smin, smax = (int(min(sh)), int(max(sh))) if C else (0, 0)
    nat.call("sglm_lag_valid_rows", nat.ptr(Xbig), T, P, Xbig.shape[1], nat.ptr(s_d) if C else None,
             nat.ptr(h_d) if C else None, C, smin, smax, int(fill_is_nan), nat.ptr(valid), nat.ptr(summ), _st())
    return _host(valid), _host(summ)


def _lag_cases(T, P):
    mixed = ([0, 1, 2, 0, 2, 1, 0], [0, 3, -2, -7, 11, 1, 25])
    return {"mixed": mixed, "positive": ([2, 0, 1, 1], [1, 9, 4, 30]), "negative": ([1, 0, 2], [-1, -12, -5]),
            "|shift| >= T": ([0, 1, 2], [T, -T - 3, 2]), "no columns": ([], []),
            "one column": ([P - 2], [0])}


@pytest.mark.parametrize("T", [5000, 600_000])
@pytest.mark.parametrize("fill_is_nan", [1, 0])
def test_lag_valid_rows(T, fill_is_nan):
    """valid[t] = 1 when row t of the lag design holds no NaN; NaN in rows 0 and T - 1 of read columns and in the
    base column 3 that no design column reads (it must not invalidate a row); ldx > P with NaN padding; bytes past
    T untouched; summary3 = {count, first, last}."""
    P = 4
    rng = np.random.default_rng(T + fill_is_nan)
    X = rng.standard_normal((T, P))
    X[0, 0] = X[T - 1, 2] = np.nan
    X[rng.integers(0, T, 5), 1] = np.nan
    X[rng.integers(0, T, 50), 3] = np.nan
    Xbig, _ = _padded(X, P + 3, np.nan)
    for what, (src, sh) in _lag_cases(T, P).items():
        valid, summ = _lag_valid(Xbig, X, src, sh, fill_is_nan)
        want = ref.lag_valid(X, src, sh, bool(fill_is_nan))
        assert np.array_equal(valid[:T], want.astype(np.uint8)), what
        assert (valid[T:] == 0xA5).all(), what
        assert np.array_equal(summ, ref.lag_summary(want)), (what, summ)


def test_lag_valid_rows_empty():
    Xbig = torch.zeros((1, 4), dtype=F64, device="cuda")
    valid, summ = _lag_valid(Xbig, np.zeros((0, 4)), [0, 1], [1, -1], 1)
    assert summ.tolist() == [0, 0, -1] and (valid == 0xA5).all()


# --------------------------------------------------------------------------- gathers
NAN_PAYLOAD = np.array([0x7FF8DEADBEEF0001], dtype=np.uint64).view(np.float64)[0]


@pytest.mark.parametrize("fill", [NAN_PAYLOAD, -0.0, np.nan], ids=["nan payload", "-0.0", "nan"])
def test_timeshift_rows(fill):
    """out[r, c] = X[rows[r] - shift_c, src_c] or fill, for sorted, unsorted and repeated row lists that include
    rows 0 and T - 1; ldo > C with sentinel padding that must survive; ldx > P."""
    T, P = 3000, 5
    rng = np.random.default_rng(5)
    X = rng.standard_normal((T, P))
    X[7, 1] = np.nan
    Xbig, _ = _padded(X, P + 2, 1e300)
    src = np.array([0, 1, 4, 4, 2, 3, 1, 0, 2], np.int32)
    sh = np.array([0, 1, -1, 40, -40, 2999, -3000, 3, 7], np.int32)
    C = len(src)
    full = ref.gather(X, src, sh, fill)
    pick = rng.random(T) < 0.5
    pick[[0, T - 1]] = True
    srt = np.flatnonzero(pick)
    lists = {"sorted": srt, "unsorted": rng.permutation(srt), "repeated": np.concatenate([srt[:50], srt[:50], [0, 0]])}
    for what, rows in lists.items():
        out = torch.full((len(rows), C + 3), SENT_F, dtype=F64, device="cuda")
        rd, src_d, sh_d = _dev(rows.astype(np.int64)), _dev(src), _dev(sh)      # held: the call takes raw pointers
        nat.call("sglm_timeshift_rows_f64", nat.ptr(Xbig), T, P, P + 2, nat.ptr(src_d), nat.ptr(sh_d), C,
                 nat.f64_bits(fill), nat.ptr(rd), len(rows), nat.ptr(out), C + 3, _st())
        _same_bits(out[:, :C], full[rows], what)
        assert (_bits(out[:, C:]) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all(), what


def _ts_path(T, P, C, span, smin, smax, ldo, out_ptr):
    """The host's choice in sglm_timeshift_f64_ranged: (tile rows or 0 = direct kernel, 16-byte stores)."""
    if smax >= T or -smin >= T:
        return 0, False
    off_bytes = (C + 1) // 2 * 2 * 4
    for tr in (64, 32, 16, 8):
        if off_bytes + (tr + span) * P * 8 <= 160 * 1024:
            return tr, C % 2 == 0 and ldo % 2 == 0 and out_ptr % 16 == 0
    return 0, False


# (what, P, C, span, smin, T values, ldo extra, out 8 bytes past a 16-byte boundary, want tile, want 16-byte)
GATHER_PLANS = [
    ("staged 16B tile64", 8, 40, 20, -10, [63, 65, 1000], 0, False, 64, True),
    ("staged 8B odd C", 8, 41, 20, -10, [65, 1000], 0, False, 64, False),
    ("staged 8B odd ldo", 8, 40, 20, -10, [1000], 1, False, 64, False),
    ("staged 8B offset out", 8, 40, 20, -10, [1000], 2, True, 64, False),
    ("staged tile32", 400, 40, 5, -2, [31, 33, 1000], 0, False, 32, True),
    ("staged tile16", 700, 40, 5, -3, [15, 17, 1000], 0, False, 16, True),
    ("staged tile8", 1200, 39, 5, -2, [7, 9, 1000], 0, False, 8, False),
    ("staged tile32 smin>0", 100, 38, 150, 4, [1000], 0, False, 32, True),
    ("staged tile16 smax<0", 100, 38, 180, -185, [1000], 0, False, 16, True),
    ("direct span", 100, 38, 210, -100, [1000], 0, False, 0, False),
    ("direct |shift|>=T", 8, 40, 30, -10, [20], 0, False, 0, False),
]


@pytest.mark.parametrize("plan", GATHER_PLANS, ids=[p[0] for p in GATHER_PLANS])
def test_timeshift_ranged_paths(plan):
    """The gather over the path matrix of the host code: staged with 16- or 8-byte stores, tile rows 64 / 32 / 16 /
    8, the direct kernel; T = tile +- 1; smin > 0 and smax < 0.  Each case asserts from the host formula
    off_bytes + (tile_rows + span) P 8 <= 160 KB that it lands where intended.  Reference: the C oracle's gather.
    The padding of X holds a value no design column may show; the padding of out must survive."""
    what, P, C, span, smin, Ts, ld_extra, offset, want_tile, want_vec = plan
    rng = np.random.default_rng(C + span)
    smax = smin + span
    src = rng.integers(0, P, C).astype(np.int32)
    sh = rng.integers(smin, smax + 1, C).astype(np.int32)
    sh[:2] = [smin, smax]
    for T in Ts:
        X = rng.standard_normal((T, P))
        X[rng.integers(0, T, 3), rng.integers(0, P, 3)] = np.nan
        Xbig, _ = _padded(X, P + 1, -1.25e300)
        ldo = C + ld_extra
        raw = torch.full((T * ldo + 4,), SENT_F, dtype=F64, device="cuda")
        base = 1 if offset else 0
        if offset:
            assert raw[1:].data_ptr() % 16 == 8
        out = raw[base: base + T * ldo].view(T, ldo)
        tile, vec = _ts_path(T, P, C, span, smin, smax, ldo, out.data_ptr())
        assert (tile, vec) == (want_tile, want_vec), (what, T, tile, vec)
        src_d, sh_d = _dev(src), _dev(sh)                                 # held: the call takes raw pointers
        nat.call("sglm_timeshift_f64_ranged", nat.ptr(Xbig), T, P, P + 1, nat.ptr(src_d), nat.ptr(sh_d), C,
                 smin, smax, nat.NAN_BITS, nat.ptr(out), ldo, _st())
        _same_bits(out[:, :C], orc.timeshift_c(X, src, sh, np.nan), f"{what} T={T}")
        rest = torch.cat([raw[:base], out[:, C:].reshape(-1), raw[base + T * ldo:]])
        assert (_bits(rest) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all(), (what, T, "padding written")


# --------------------------------------------------------------------------- roll, crop
@pytest.mark.parametrize("n", [1, 2, 257, 1 << 20])
def test_roll(n):
    x = np.random.default_rng(n).standard_normal(n)
    xd = _dev(x)
    for shift in (0, 1, -1, n, -n, n + 3, -(2 * n + 1), (1 << 40) + 5):
        out = torch.full((n + 8,), SENT_F, dtype=F64, device="cuda")
        nat.call("sglm_roll_f64", nat.ptr(xd), n, shift, nat.ptr(out), _st())
        _same_bits(out[:n], np.roll(x, shift), f"roll n={n} shift={shift}")
        assert (_bits(out[n:]) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all()


def test_crop_rows():
    T, C = 5000, 13
    X = np.random.default_rng(2).standard_normal((T, C))
    Xbig, _ = _padded(X, C + 3, np.nan)
    for begin, n, cols in [(0, T, C), (17, 500, C), (T - 1, 1, 5), (4095, 905, 1)]:
        out = torch.full((n, C + 2), SENT_F, dtype=F64, device="cuda")
        nat.call("sglm_crop_rows_f64", nat.ptr(Xbig), C + 3, begin, n, cols, nat.ptr(out), C + 2, _st())
        _same_bits(out[:, :cols], X[begin: begin + n, :cols], f"crop {begin} {n} {cols}")
        assert (_bits(out[:, cols:]) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all()


# --------------------------------------------------------------------------- column moments
def _moment_columns(T, C, rng, skipna, special):
    X = rng.standard_normal((T, C)) * np.exp2(rng.integers(-8, 9, C)) + rng.uniform(-50, 50, C)
    if not special:
        return X
    k = 0
    if C > 5:
        X[:, 0] = np.nan                                       # all NaN
        X[:, 1] = np.nan
        X[T // 2, 1] = 3.75                                    # one non-NaN entry
        X[:, 2] = 0.1                                          # constant (0.1 is not a binary fraction)
        X[:, 3] = 1e8 + rng.standard_normal(T)                 # large mean: a one-pass formula fails
        X[:, 4] = rng.choice([-1.0, 1.0], T) * np.exp2(rng.integers(-30, 31, T))        # 60 binades
        k = 5
    if T > 2 and C > k + 1:
        X[rng.integers(0, T, 3), k] = np.nan                  # propagates (numpy) or is skipped (pandas)
    return X


MOMENT_PLANS = [(1, 1, 0), (1, 7, 2), (2, 7, 0), (CH, 256, 1), (CH + 1, 257, 3), (3 * CH + 5, 600, 2),
                (300_000, 3, 1), (300_000, 8, 0)]


@pytest.mark.parametrize("T,C,ld_extra", MOMENT_PLANS)
@pytest.mark.parametrize("ddof,skipna", [(0, 0), (1, 1), (0, 1), (1, 0)])
def test_col_moments(T, C, ld_extra, ddof, skipna):
    """Mean and sd within bounds (1) and (3) of the module docstring; NaN exactly where the reference is NaN (an
    all-NaN column gives NaN for both, a single value with ddof 1 a NaN sd); repeated calls give the same bits;
    NaN in the ldx padding is never read."""
    rng = np.random.default_rng(T * 3 + C + ddof + 2 * skipna)
    X = _moment_columns(T, C, rng, skipna, special=True)
    Xbig, _ = _padded(X, C + ld_extra, np.nan)
    wb = nat.lib().sglm_col_moments_workspace_bytes(T, C)
    ws = torch.empty(wb // 8 + 1, dtype=F64, device="cuda")
    res = []
    for _ in range(2):
        mean = torch.full((C,), SENT_F, dtype=F64, device="cuda")
        sd = torch.full((C,), SENT_F, dtype=F64, device="cuda")
        nat.call("sglm_col_moments_f64", nat.ptr(Xbig), C + ld_extra, T, C, ddof, skipna, nat.ptr(mean), nat.ptr(sd),
                 nat.ptr(ws), wb, _st())
        res.append((_host(mean), _host(sd)))
    _same_bits(res[0][0], res[1][0], "mean: repeated call")
    _same_bits(res[0][1], res[1][1], "sd: repeated call")
    m_gpu, s_gpu = res[0]
    m_ref, s_ref, n, absum = ref.col_moments(X, ddof, skipna)
    assert np.array_equal(np.isnan(m_gpu), np.isnan(m_ref.astype(np.float64))), "mean NaN positions"
    assert np.array_equal(np.isnan(s_gpu), np.isnan(s_ref.astype(np.float64))), "sd NaN positions"
    L, K = min(T, CH), -(-T // CH)
    fin = ~np.isnan(m_ref)
    with np.errstate(invalid="ignore", divide="ignore"):
        bm = 2 * (L + K) * U * absum / n                                                              # (1)
    dm = np.abs(m_gpu.astype(LD) - m_ref)
    assert np.all(dm[fin] <= bm[fin]), ("mean", np.flatnonzero(fin & (dm > bm))[:5], dm[fin].max())
    fs = ~np.isnan(s_ref)
    if not fs.any():
        return
    var = s_ref[fs] ** 2
    nn = n[fs].astype(LD)
    Qm = var * (nn - ddof) + nn * dm[fs] ** 2                                                           # Q(m)
    bv = (2 * (L + K + 4) * U * Qm + nn * dm[fs] ** 2) / (nn - ddof)                                    # (2)
    with np.errstate(divide="ignore", invalid="ignore"):
        bs = (np.minimum(np.sqrt(bv), np.where(s_ref[fs] > 0, bv / s_ref[fs], np.inf))
              + 2 * U * (s_ref[fs] + np.sqrt(bv)))                                                      # (3)
    ds = np.abs(s_gpu[fs].astype(LD) - s_ref[fs])
    assert np.all(ds <= bs), ("sd", np.flatnonzero(fs)[ds > bs][:5], (ds / bs).max())


def test_col_moments_large_mean_needs_two_passes():
    """The 1e8 + N(0, 1) column: the bound (3) is far below what sum x^2 / n - mean^2 can deliver."""
    T = 3 * CH + 5
    rng = np.random.default_rng(9)
    X = (1e8 + rng.standard_normal(T))[:, None]
    Xd = _dev(X)
    wb = nat.lib().sglm_col_moments_workspace_bytes(T, 1)
    ws = torch.empty(wb // 8 + 1, dtype=F64, device="cuda")
    mean = torch.empty(1, dtype=F64, device="cuda")
    sd = torch.empty(1, dtype=F64, device="cuda")
    nat.call("sglm_col_moments_f64", nat.ptr(Xd), 1, T, 1, 0, 0, nat.ptr(mean), nat.ptr(sd), nat.ptr(ws), wb, _st())
    one_pass = np.sqrt(max(np.mean(X * X) - np.mean(X) ** 2, 0.0))
    s_ref = float(ref.col_moments(X, 0, 0)[1][0])
    assert abs(sd.item() - s_ref) < 1e-6 * s_ref
    assert abs(one_pass - s_ref) > 1e-3 * s_ref


# --------------------------------------------------------------------------- z-score, diff
def test_zscore_apply():
    """(x - mean) / sd bit for bit against numpy with test-supplied moments: sd = 0, +-inf and NaN inputs, NaN mean;
    ldx > C and ldo > C, the out padding left alone."""
    T, C = 4097, 9
    rng = np.random.default_rng(4)
    X = rng.standard_normal((T, C)) * 3 + 1
    X[5, :] = np.inf
    X[6, :] = -np.inf
    X[7, :] = np.nan
    X[8, :] = 0.0
    mean = rng.standard_normal(C)
    sd = np.abs(rng.standard_normal(C)) + 0.1
    sd[0], sd[1], sd[2], mean[3] = 0.0, np.inf, np.nan, np.nan
    X[9, 0] = mean[0]                                            # 0 / 0
    Xbig, _ = _padded(X, C + 2, np.nan)
    out = torch.full((T, C + 3), SENT_F, dtype=F64, device="cuda")
    mean_d, sd_d = _dev(mean), _dev(sd)
    nat.call("sglm_zscore_apply_f64", nat.ptr(Xbig), C + 2, T, C, nat.ptr(mean_d), nat.ptr(sd_d), nat.ptr(out),
             C + 3, _st())
    with np.errstate(all="ignore"):
        want = ref.zscore(X, mean, sd)
    got = _host(out[:, :C])
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    _same_bits(got[~nan], want[~nan], "zscore")
    assert (_bits(out[:, C:]) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all()


@pytest.mark.parametrize("T", [1, 2, 4097])
@pytest.mark.parametrize("cols", [None, [4, 2, 2, 0], [5, 4, 3, 2, 1, 0]], ids=["all", "repeats", "reversed"])
def test_diff1(T, cols):
    """out[t][j] = X[t + 1][cols[j]] - X[t][cols[j]]: np.diff's bits on finite values, NaN where np.diff is NaN;
    ldx / ldo padding; T = 1 writes nothing."""
    C = 6
    rng = np.random.default_rng(T)
    X = rng.standard_normal((T, C)) * np.exp2(rng.integers(-20, 21, (T, C)))
    if T > 10:
        X[3, 1], X[4, 2], X[5, 2] = np.nan, np.inf, np.inf
    sel = list(range(C)) if cols is None else cols
    Xbig, _ = _padded(X, C + 1, np.nan)
    ldo = len(sel) + 2
    out = torch.full((max(T - 1, 1), ldo), SENT_F, dtype=F64, device="cuda")
    cd = _dev(np.asarray(sel, np.int32)) if cols is not None else None
    nat.call("sglm_diff1_f64", nat.ptr(Xbig), C + 1, T, nat.ptr(cd), len(sel), nat.ptr(out), ldo, _st())
    if T == 1:
        assert (_bits(out) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all()
        return
    with np.errstate(invalid="ignore"):
        want = np.diff(X[:, sel], axis=0)
    got = _host(out[:, :len(sel)])
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    _same_bits(got[~nan], want[~nan], "diff1")
    assert (_bits(out[:, len(sel):]) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all()


# --------------------------------------------------------------------------- rolling 5-95 % min-max
ROLL_W = [2, 3, 4, 5, 20, 21, 40, 255, 256, 257, 513, 1000, 4096, 16384]


def _rolling(x, W, seg=None):
    xd = _dev(x)
    out = torch.full((len(x) + 8,), SENT_F, dtype=F64, device="cuda")
    lo = hi = None
    if seg is not None:
        lo, hi = _dev(seg[0].astype(np.int64)), _dev(seg[1].astype(np.int64))
    nat.call("sglm_rolling_minmax_f64", nat.ptr(xd), len(x), nat.ptr(lo), nat.ptr(hi), W, nat.ptr(out), _st())
    assert (_bits(out[len(x):]) == np.uint64(SENT & 0xFFFFFFFFFFFFFFFF)).all(), "written past n"
    return _host(out[:len(x)])


def _roll_series(kind, n, rng):
    if kind == "walk":
        return np.cumsum(rng.standard_normal(n))
    if kind == "events":                                       # 0/1 ties, constant windows (0 / 0 = NaN)
        return (rng.random(n) < 0.1).astype(np.float64)
    x = np.cumsum(rng.standard_normal(n))
    if kind == "nan":
        x[rng.choice(n, max(n // 500, 2), replace=False)] = np.nan
    elif kind == "inf":
        x[rng.choice(n, 2, replace=False)] = np.inf
        x[rng.choice(n, 2, replace=False)] = -np.inf
    elif kind == "flat":                                       # a constant stretch longer than the window
        x[n // 3: n // 3 + n // 4] = 2.5
    return x


@pytest.mark.parametrize("W", ROLL_W)
def test_rolling_minmax(W):
    """Equal to the reference: n < W (all NaN), n = W (one valid position), n > 8 SMs (the grid-stride loop);
    NaN inside windows, ties, +-inf (pandas counts them as missing), constant windows; segments shorter than W,
    of exactly W and longer, so windows touch both segment ends."""
    rng = np.random.default_rng(W)
    n = max(3000, 8 * _sms() + 200) + (W if W > 1000 else 2 * W)
    kinds = ["walk", "events", "nan", "inf", "flat"] if W <= 1000 else ["walk", "nan"]
    for kind in kinds:
        x = _roll_series(kind, n, rng)
        _same_values(_rolling(x, W), ref.rolling_minmax(x, W), f"W={W} {kind}")
    for m in (W - 1, W):
        x = _roll_series("walk", m, rng)
        _same_values(_rolling(x, W), ref.rolling_minmax(x, W), f"W={W} n={m}")
    if W <= 1000:
        sizes = [W - 1, 1, W, W + 1, 3 * W + 7, 500]
        x = _roll_series("nan", sum(sizes), rng)
        seg = ref.segments_of(sizes)
        _same_values(_rolling(x, W, seg), ref.rolling_minmax(x, W, *seg), f"W={W} segments")


@pytest.mark.parametrize("grouped", [False, True])
def test_detrend_data_device_equals_host(grouped):
    """detrend_data(device=True) returns pandas' Series bit for bit (values and index), grouped and ungrouped."""
    rng = np.random.default_rng(int(grouped))
    n = 2400
    df = pd.DataFrame({"v": np.cumsum(rng.standard_normal(n)), "g": rng.integers(0, 4, n)})
    df.loc[rng.choice(n, 3, replace=False), "v"] = np.nan
    cols = ["g"] if grouped else []
    for w in (10, 20):
        want = sglm_pp.detrend_data(df, "v", cols, w, device=False)
        got = sglm_pp.detrend_data(df, "v", cols, w, device=True)
        assert got.index.equals(want.index)
        _same_values(got.to_numpy(), want.to_numpy(), f"detrend w={w} grouped={grouped}")
