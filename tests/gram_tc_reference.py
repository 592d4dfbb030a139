"""Bit-exact CPU model of the tensor-core Gram (csrc/gram_tc.cu) and longdouble references of the fp64 statistics
kernels (csrc/suffstats.cu, csrc/solvers.cu, csrc/poisson_batch.cu).  numpy only.

The tensor-core Gram, as its comments specify it, for Z = [X | Y | 1] (optionally every row scaled by rs[t]):

  analysis      v = |z * rs| (one fp64 product); colmax = max v, lsb = lowest set bit of any v (IEEE fields,
                subnormals included); E = ilogb(colmax) + 1 (0 for an all-zero column), S = 1 + (span + 6) // 7 with
                span = E - 6 - lsb (S = 1 when span <= 0), capped at max_planes;
  slicing       r = z * 2^(6 - E) (one multiplication by a power of two when |E| < 900, else ldexp(z, -E) * 64, which
                rounds twice when ldexp's result is subnormal), then S times  d_k = rint(r), r = (r - d_k) * 128;
  plane Grams   SG[(c1, k), (c2, l)] = sum over the set's rows of d_k(c1) d_l(c2): exact integers;
  recombination for tot = 9 down to 2: part = sum of the plane Grams with k + l = tot in ascending k,
                acc += ldexp(part, -(12 + 7 (tot - 2)));  G = ldexp(acc, E1 + E2), upper triangle mirrored.
                Pairs with k + l > 9 are dropped.

The plane Grams are computed with a float64 matmul of the digits: every product is at most 2^12 and every partial sum
at most T 2^12 < 2^53, so any summation order gives the exact integer, and the model costs one numpy GEMM."""
import numpy as np

SMAX = 8                      # TC_SMAX: digit planes of a general fp64 column
TC_BK, TC_BM, TC_BN = 128, 256, 256
TC_MAX_KB_PER_SEG = 2048      # 2048 * 128 rows * 2^12 = 2^30: int32 accumulators drained per segment
FAST_E = 900                  # |E| < 900: scaling by one exact power-of-two multiplication
EMPTY_LSB = 0x7F7F7F7F        # col_lsb of a column without a non-zero value (the kernels' memset pattern)
NAN_BITS = 0x7FF8000000000000
DBL_MAX = np.finfo(np.float64).max

LD = np.longdouble
U = 2.0 ** -53


def augment(X, Y):
    """Z = [X | Y | 1] as a float64 array [T][C + n_y + 1]."""
    X = np.asarray(X, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    Y = Y.reshape(len(Y), -1) if Y.ndim == 1 else Y
    return np.concatenate([X, Y, np.ones((X.shape[0], 1))], axis=1)


def _scaled(Z, rs):
    Z = np.asarray(Z, dtype=np.float64)
    if rs is None:
        return Z
    with np.errstate(over="ignore", invalid="ignore"):
        return Z * np.asarray(rs, dtype=np.float64)[:, None]


def _lsb(v):
    """Exponent of the lowest set bit of each non-negative double (v = m 2^e with m odd); EMPTY_LSB for zeros.
    Non-finite values count with their IEEE fields, as in tc_colmax_kernel (their columns are flagged anyway)."""
    bits = np.ascontiguousarray(v, dtype=np.float64).view(np.uint64)
    e = (bits >> np.uint64(52)).astype(np.int64)
    frac = bits & np.uint64((1 << 52) - 1)
    m = np.where(e > 0, frac | np.uint64(1 << 52), frac)
    low = m & (~m + np.uint64(1))                              # lowest set bit of the significand
    with np.errstate(divide="ignore"):
        tz = np.where(m > 0, np.log2(np.maximum(low, np.uint64(1)).astype(np.float64)), 0).astype(np.int64)
    out = np.where(e > 0, e - 1075 + tz, -1074 + tz)
    return np.where(m > 0, out, EMPTY_LSB)


def colstats(Z, rs=None):
    """(colmax_bits uint64, col_lsb int32) of tc_colmax_kernel: the bits of max |z rs| per column (the NaN pattern when
    a value is NaN or inf; 0 for no rows) and the lowest set bit of any value (EMPTY_LSB when there is none)."""
    with np.errstate(invalid="ignore"):
        v = np.abs(_scaled(Z, rs))
    n_aug = v.shape[1]
    if v.shape[0] == 0:
        return np.zeros(n_aug, dtype=np.uint64), np.full(n_aug, EMPTY_LSB, dtype=np.int32)
    bad = ~np.all(v <= DBL_MAX, axis=0)
    m = np.max(np.where(np.isnan(v), 0.0, v), axis=0)
    bits = np.ascontiguousarray(m).view(np.uint64).copy()
    bits[bad] = NAN_BITS
    return bits, np.min(_lsb(v), axis=0).astype(np.int32)


def exponents(colmax_bits, col_lsb, max_planes=SMAX):
    """(colE, colS, flag) of tc_exponent_kernel."""
    m = np.ascontiguousarray(colmax_bits, dtype=np.uint64).view(np.float64)
    lsb = np.asarray(col_lsb, dtype=np.int64)
    bad = ~(m <= DBL_MAX)
    mm = np.where(bad, 0.0, m)
    E = np.where(mm == 0.0, 0, np.frexp(mm)[1]).astype(np.int64)       # frexp: m = f 2^e, 0.5 <= f < 1 -> e = ilogb + 1
    span = E - 6 - lsb
    need = np.where((mm != 0.0) & (span > 0), 1 + (span + 6) // 7, 1)
    S = np.minimum(need, max_planes)
    E = np.where(bad, 0, E)
    S = np.where(bad, 1, S)
    return E.astype(np.int32), S.astype(np.int32), int(bad.any())


def analyze(Z, rs=None, max_planes=SMAX):
    """-> dict(colmax_bits, col_lsb, colE, colS, flag) of sglm_gram_tc_analyze(_scaled)_f64."""
    bits, lsb = colstats(Z, rs)
    E, S, flag = exponents(bits, lsb, max_planes)
    return dict(colmax_bits=bits, col_lsb=lsb, colE=E, colS=S, flag=flag)


def _first_remainder(z, E):
    """r = z 2^(6 - E) as tc_slice_kernel computes it (both branches)."""
    with np.errstate(over="ignore", under="ignore", invalid="ignore"):
        if -FAST_E < E < FAST_E:
            return z * np.ldexp(1.0, 6 - int(E))
        return np.ldexp(z, -int(E)) * 64.0


def digits(Z, rs, colE, colS):
    """int8 digit planes per column: a list of [S_c][T] arrays (np.rint is round-half-even like CUDA rint)."""
    Zs = _scaled(Z, rs)
    out = []
    for c in range(Zs.shape[1]):
        r = _first_remainder(Zs[:, c], colE[c])
        planes = np.empty((int(colS[c]), Zs.shape[0]), dtype=np.int8)
        for k in range(int(colS[c])):
            d = np.rint(r)
            r = (r - d) * 128.0
            planes[k] = d.astype(np.int8)
        out.append(planes)
    return out


def digits_needed(z, E):
    """Planes (1..8) the digit-by-digit expansion of one value needs at scale 2^E (tc_digits_kernel's count, which
    is 8 also when 8 planes do not suffice)."""
    r = np.ldexp(np.float64(z), -int(E)) * 64.0
    need = 0
    for k in range(1, SMAX + 1):
        if r == 0.0:
            break
        d = np.rint(r)
        if d != 0.0:
            need = k
        r = (r - d) * 128.0
    return SMAX if r != 0.0 else need


def _stack(planes):
    """All planes as one float64 matrix [sum S_c][T] and the row of plane k (1-based) of column c (-1: none)."""
    idx = np.full((len(planes), SMAX), -1, dtype=np.int64)
    rows, n = [], 0
    for c, p in enumerate(planes):
        idx[c, :p.shape[0]] = np.arange(n, n + p.shape[0])
        n += p.shape[0]
        rows.append(p)
    A = np.concatenate(rows, axis=0).astype(np.float64) if rows else np.zeros((0, 0))
    return A, idx


def plane_grams(planes, rows):
    """Exact int64 Grams of all digit planes over the row indices `rows` -> (SG [P][P], plane index [n_aug][8])."""
    A, idx = _stack(planes)
    rows = np.asarray(rows, dtype=np.int64)
    assert len(rows) * 4096 < 2 ** 53, "plane Gram would not be exact in float64"
    At = A[:, rows]
    SG = At @ At.T
    return SG.astype(np.int64), idx


def combine(SG, idx, colE, colS):
    """tc_combine_kernel: fp64 recombination of the plane Grams, vectorised over the column pairs."""
    n = len(colE)
    S = np.asarray(colS, dtype=np.int64)
    SGz = np.zeros((SG.shape[0] + 1, SG.shape[0] + 1))
    SGz[:-1, :-1] = SG                                  # index -1 -> the zero row / column
    acc = np.zeros((n, n))
    for tot in range(SMAX + 1, 1, -1):                  # smallest weights first
        part = np.zeros((n, n))
        for k in range(1, SMAX + 1):                    # ascending k
            l = tot - k
            if l < 1 or l > SMAX:
                continue
            ok = (S[:, None] >= k) & (S[None, :] >= l)
            v = SGz[idx[:, k - 1][:, None], idx[:, l - 1][None, :]]
            part = part + np.where(ok, v, 0.0)
        acc = acc + np.ldexp(part, -(12 + 7 * (tot - 2)))
    Es = np.asarray(colE, dtype=np.int64)
    with np.errstate(over="ignore"):
        G = np.ldexp(acc, (Es[:, None] + Es[None, :]).astype(np.int32))
    iu = np.triu(np.ones((n, n), dtype=bool))
    return np.where(iu, G, G.T)                         # the kernel computes c1 <= c2 and mirrors


def gram_with(Z, colE, colS, sets, rs=None):
    """G [n_sets][n_aug][n_aug] from a given analysis (the lag design supplies its own)."""
    planes = digits(Z, rs, colE, colS)
    out = []
    for rows in sets:
        SG, idx = plane_grams(planes, rows)
        out.append(combine(SG, idx, colE, colS))
    return np.stack(out) if out else np.zeros((0, Z.shape[1], Z.shape[1]))


def gram(Z, sets, rs=None, max_planes=SMAX):
    """-> (G [n_sets][n_aug][n_aug], analysis dict).  sets: row-index arrays."""
    a = analyze(Z, rs, max_planes)
    return gram_with(Z, a["colE"], a["colS"], sets, rs), a


def lag_design(base, src, off, T):
    """Z[t, c] = base[t + off[c], src[c]] for t < T."""
    base = np.asarray(base, dtype=np.float64)
    t = np.arange(T)[:, None]
    return base[t + np.asarray(off)[None, :], np.asarray(src)[None, :]]


def lag_analysis(base, src, Y):
    """_engine._lag_analysis: exponents / planes of [base | 1] over the window; a lag column takes those of its base
    signal, the response and ones columns those of [Y | 1]."""
    b = analyze(augment(base, np.zeros((base.shape[0], 0))))
    y = analyze(augment(np.zeros((Y.shape[0], 0)), Y))
    src = np.asarray(src)
    colE = np.concatenate([b["colE"][src], y["colE"]]).astype(np.int32)
    colS = np.concatenate([b["colS"][src], y["colS"]]).astype(np.int32)
    return colE, colS, b["colE"], b["colS"]


def lag_gram(base, src, off, Y, sets):
    """Gram of the lag design [base[t + off_c, src_c] | Y | 1] with the lag analysis."""
    Y = np.asarray(Y, dtype=np.float64).reshape(len(Y), -1)
    colE, colS, _, _ = lag_analysis(base, src, Y)
    Z = augment(lag_design(base, src, off, Y.shape[0]), Y)
    return gram_with(Z, colE, colS, sets), colE, colS


def plan(n_aug, colS, set_rows, sms=148):
    """tc_make_plan: level-major plane rows (each level padded to 256), the 256 x 256 output tiles (level pairs
    k <= l with k + l <= 9, upper triangle inside a level), the 2-CTA pairs, the K parts and the K segments."""
    colS = np.asarray(colS)
    plane_row = np.full((n_aug, SMAX), -1, dtype=np.int64)
    level_off, level_cnt = [0] * (SMAX + 1), [0] * (SMAX + 1)
    off = 0
    for k in range(1, SMAX + 1):
        level_off[k] = off
        cols = np.flatnonzero(colS >= k)
        plane_row[cols, k - 1] = off + np.arange(len(cols))
        level_cnt[k] = len(cols)
        off += (len(cols) + 255) // 256 * 256
    S = max(off, 256)
    tiles, tile_levels = [], []
    for k in range(1, SMAX + 1):
        for l in range(k, SMAX + 1):
            if k + l > SMAX + 1 or not level_cnt[k] or not level_cnt[l]:
                continue
            mt0, mt1 = level_off[k] // TC_BM, (level_off[k] + level_cnt[k] + TC_BM - 1) // TC_BM
            nt0, nt1 = level_off[l] // TC_BN, (level_off[l] + level_cnt[l] + TC_BN - 1) // TC_BN
            for mt in range(mt0, mt1):
                for nt in range(nt0, nt1):
                    if k == l and (nt + 1) * TC_BN <= mt * TC_BM:
                        continue
                    tiles.append((mt, nt))
                    tile_levels.append((k, l))
    pairs, i = [], 0
    while i < len(tiles):
        if i + 1 < len(tiles) and tiles[i + 1][0] == tiles[i][0] and tiles[i + 1][1] == tiles[i][1] + 1:
            pairs.append((i, i + 1))
            i += 2
        else:
            pairs.append((i, -1))
            i += 1
    nt_items = max(1, 2 * len(pairs))
    total_kb = sum((int(r) + TC_BK - 1) // TC_BK for r in set_rows)
    best, best_eff = 1, 0.0
    for parts in range(1, 17):
        if parts > 1 and total_kb // parts < 64:
            break
        items = nt_items * parts
        eff = items / (((items + sms - 1) // sms) * sms)
        score = eff - (0.5 if items < 2 * sms else 0.0) - 0.002 * parts
        if score > best_eff:
            best_eff, best = score, parts
    segs, pos = [], 0
    for s, r in enumerate(set_rows):
        kb, kb0 = (int(r) + TC_BK - 1) // TC_BK, pos // TC_BK
        if kb == 0:
            segs.append((kb0, 0, s))
        while kb > 0:
            n = min(kb, TC_MAX_KB_PER_SEG)
            segs.append((kb0, n, s))
            kb0 += n
            kb -= n
        pos += (int(r) + TC_BK - 1) // TC_BK * TC_BK
    return dict(S=S, n_pos=max(pos, TC_BK), tiles=tiles, tile_levels=tile_levels, pairs=pairs, n_parts=best,
                segs=segs, plane_row=plane_row, level_off=level_off, level_cnt=level_cnt)


# --------------------------------------------------------------------------- inputs
def catalogue(T, rng):
    """Adversarial columns (name -> [T] float64) for the digit slicing, used as columns of X and of Y."""
    t = np.arange(T)
    cols = {}
    cols["pow2_pos"] = np.where(t % 5 == 0, 2.0 ** 10, rng.uniform(-1, 1, T) * 2.0 ** 9)
    cols["pow2_neg_max"] = np.where(t % 7 == 3, -2.0 ** -3, rng.uniform(-1, 1, T) * 2.0 ** -5)
    E = 4
    cols["first_digit_64"] = np.where(t % 3 == 0, (1 - 2.0 ** -8) * 2.0 ** E, -(1 - 2.0 ** -8) * 2.0 ** E)
    # round-half-even ties at planes 1, 2, 3 and 4 (E = 0: r = 64 z); a tie at plane k leaves a digit of +-64 at k + 1
    q = 1.0 / 128
    ties = np.array([2.5, -2.5, 3.5, 2 + 3.5 * q, -(2 + 3.5 * q), 5 + (1 + 6.5 * q) * q, -(7 + (3 + (2 + 0.5 * q) * q) * q),
                     64 * (1 - 2.0 ** -8)]) / 64
    cols["ties"] = ties[t % len(ties)]
    cols["zero_one"] = (rng.random(T) < 0.2).astype(np.float64)
    cols["small_int"] = rng.integers(-40, 41, T).astype(np.float64)
    cols["dyadic"] = rng.integers(-1000, 1000, T) * 2.0 ** -9
    neg0 = np.where(t % 4 == 0, -0.0, rng.uniform(0, 1, T))
    cols["neg_zero"] = neg0
    cols["all_zero"] = np.where(t % 2 == 0, 0.0, -0.0)
    cols["constant"] = np.full(T, 3.0)
    cols["one_plus_tiny"] = np.where(t % 3 == 0, 1.0, 2.0 ** -60)
    cols["one_plus_ulp"] = np.where(t % 2 == 0, 1.0 + 2.0 ** -52, 0.75)
    cols["subnormal_mix"] = np.where(t % 3 == 0, 5e-324 * (t + 1), rng.uniform(-1, 1, T) * 2.0 ** -1000)
    cols["all_subnormal"] = (rng.integers(-2 ** 40, 2 ** 40, T)).astype(np.float64) * 5e-324
    for e in (899, 900, 901, -899, -900, -901):
        # column maximum just below 2^e: E = e (|z| < 2^E), the two sides of the |E| < 900 switch of tc_slice_kernel
        cols[f"e{e}"] = np.where(t == T // 2, (1 - 2.0 ** -30) * 2.0 ** e, rng.uniform(-1, 1, T) * 2.0 ** (e - 3))
    for e in (-1017, -1016, -1020):
        cols[f"e{e}"] = np.where(t == 1, 2.0 ** e, rng.uniform(-1, 1, T) * 2.0 ** (e - 2))
    cols["near_dbl_max"] = rng.uniform(0.5, 1.0, T) * DBL_MAX * np.where(t % 2 == 0, 1.0, -1.0)
    cols["gauss"] = rng.standard_normal(T)
    return cols


# --------------------------------------------------------------------------- longdouble references of the fp64 kernels
# Each returns (ref, mag): the longdouble value and the sum of the magnitudes of the terms it adds.  A kernel result
# passes when |got - ref| <= C_ULP * n * u * mag, n = the longest chain of fp64 roundings a term passes through
# (given next to each test).
def suffstats_dmma(Z, w=None):
    """Z' diag(w) Z (unit weights when w is None)."""
    Zl = np.asarray(Z, dtype=np.float64).astype(LD)
    wl = np.ones(Zl.shape[0], dtype=LD) if w is None else np.asarray(w, dtype=np.float64).astype(LD)
    Zw = Zl * wl[:, None]
    return Zw.T @ Zl, np.abs(Zw).T @ np.abs(Zl)


def center(A_plus, A_minus, C, n_y, y_col, fit_intercept=True):
    """sglm_center_stats_f64 in longdouble from the same fp64 statistics.  -> dict of (ref, mag) pairs."""
    Ap = np.asarray(A_plus, dtype=np.float64).astype(LD)
    Am = np.zeros_like(Ap) if A_minus is None else np.asarray(A_minus, dtype=np.float64).astype(LD)
    A, Amag = Ap - Am, np.abs(Ap) + np.abs(Am)
    one, yc = C + n_y, C + y_col
    n = A[one, one]
    xbar = A[:C, one] / n if fit_intercept else np.zeros(C, dtype=LD)
    ybar = A[yc, one] / n if fit_intercept else LD(0)
    nxx = n * np.outer(xbar, xbar)
    return dict(
        Qc=(A[:C, :C] - nxx, Amag[:C, :C] + np.abs(nxx)),
        qc=(A[:C, yc] - n * xbar * ybar, Amag[:C, yc] + np.abs(n * xbar * ybar)),
        xbar=(xbar, Amag[:C, one] / abs(n) + Amag[one, one] * np.abs(xbar) / abs(n)),
        yyc=(A[yc, yc] - n * ybar * ybar, Amag[yc, yc] + abs(n * ybar * ybar)),
        ybar=(ybar, Amag[yc, one] / abs(n) + Amag[one, one] * abs(ybar) / abs(n)),
        sy=(A[yc, one], Amag[yc, one]))


def finalize(W, xbar, ybar):
    """b = ybar - xbar . w per model (rows of W).  -> (ref, mag)."""
    Wl = np.asarray(W, dtype=np.float64).astype(LD)
    xl = np.asarray(xbar, dtype=np.float64).astype(LD)
    yl = np.asarray(ybar, dtype=np.float64).astype(LD)
    return yl - np.sum(xl * Wl, axis=1), np.abs(yl) + np.sum(np.abs(xl * Wl), axis=1)


def quadform(A, V):
    """v_m' A v_m for the rows v_m of V.  -> (ref, mag)."""
    Al = np.asarray(A, dtype=np.float64).astype(LD)
    Vl = np.asarray(V, dtype=np.float64).astype(LD)
    return np.einsum("mi,ij,mj->m", Vl, Al, Vl), np.einsum("mi,ij,mj->m", np.abs(Vl), np.abs(Al), np.abs(Vl))
