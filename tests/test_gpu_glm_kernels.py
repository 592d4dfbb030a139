"""Kernel-level references for the batched log-link GLM kernels (csrc/poisson_batch.cu) and the family row passes
(csrc/predict.cu).  The solver tests compare optima, which do not move when a Fisher weight, an objective sum or a
step-control decision is wrong; here every output of an entry point is compared with the same quantity computed from
its definition in numpy longdouble (64-bit mantissa on x86-64):

  unit loss (scikit-learn's HalfTweedieLoss, log link), its eta-derivative mu^(1-p) (mu - y), the Fisher weight
  mu^(2-p), the score / deviance terms; mu^(2-p) = exp((2-p) eta) and mu^(1-p) = exp((1-p) eta) are computed
  directly, not as a product.

Tolerances are derived: a sum or dot product of n fp64 terms must satisfy |got - ref| <= C_ULP n u sum|term_i|,
u = 2^-53.  A per-element output is the case n = 1.  For a difference such as y - mu, the terms are those of the
expanded form (|y| + |mu|).  Where eta itself comes out of a dot product (the row passes), its bound is carried
through each quantity as max |q(eta +- e) - q(eta)|.

C_ULP = 16 covers the last-place errors of exp / log / pow (at most 2 ulp each), the products and reciprocals of
the family terms, and the rounding of the exp argument (1-p) eta, which costs |(1-p) eta| ulp: the inputs keep
|eta| <= 3, so that term stays below 9.

Bit-for-bit invariants: repeated calls, a model's position in the batch and its neighbours (the epilogue grid depends
on T only; the GEMMs add every element in a fixed k order), NaN in the padding columns, and the layout of X (leading
dimension, a base pointer 8 bytes off) for the fp64 GEMMs."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
if not torch.cuda.is_available():
    pytest.skip("needs a CUDA device", allow_module_level=True)

import synth_data  # noqa: E402
import _engine as eng  # noqa: E402
import _sglm_native as nat  # noqa: E402

LD = np.longdouble
U = 2.0 ** -53
C_ULP = 16
F64 = torch.float64
POWERS = [1.0, 2.0, 1.5, 3.0, 1.2, 2.5]
MAX_REF_MADDS = 2e7          # longdouble multiply-adds of one GEMM reference


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev(a, dtype=F64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)


def _st():
    return nat.stream_ptr()


def _bits(t):
    a = t.detach().cpu().numpy() if torch.is_tensor(t) else np.asarray(t)
    return np.ascontiguousarray(a).view(np.uint64 if a.dtype == np.float64 else np.uint32)


def _same_bits(a, b, what):
    assert np.array_equal(_bits(a), _bits(b)), what


def _check(got, ref, bound, what):
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got.astype(LD) - ref)
    ok = err <= bound
    if not np.all(ok):
        i = np.unravel_index(np.argmin(np.where(ok, np.inf, -(err - bound).astype(np.float64))), err.shape)
        raise AssertionError(f"{what}: {np.count_nonzero(~ok)} of {ok.size} beyond the bound; at {i}: got {got[i]!r}, "
                             f"ref {float(ref[i])!r}, err {float(err[i]):.3e}, bound {float(bound[i]):.3e}")


def _sum_bound(n, mag):
    return C_ULP * max(n, 1) * U * mag


# --------------------------------------------------------------------------- inputs
def _lag_design(T, C, seed):
    """Columns of a lag design (synth_data: sparse 0/1 events, z-scored AR(1), a ramp) at lags 0..7."""
    P = (C + 7) // 8
    base = synth_data.synth_base(T + 8, max(P, 1), seed)
    X = np.empty((T, C))
    for j in range(C):
        X[:, j] = base[(j % 8): (j % 8) + T, j // 8]
    return X


def _wide(T, C, rng):
    """Entries over 40 binades with both signs."""
    return rng.choice([-1.0, 1.0], (T, C)) * rng.uniform(1.0, 2.0, (T, C)) * np.exp2(rng.integers(-20, 21, (T, C)))


def _layouts(X):
    """The same matrix as device views with ldx = C, C + 1, C + 3 and a base pointer 8 bytes past a 16-byte boundary
    (ldx = C + 1).  Padding holds NaN: a kernel that read it would show it."""
    T, C = X.shape
    Xc = _dev(X)
    out = [("ldx=C", Xc, C)]
    for extra in (1, 3):
        big = torch.full((T, C + extra), float("nan"), dtype=F64, device="cuda")
        big[:, :C] = Xc
        out.append((f"ldx=C+{extra}", big[:, :C], C + extra))
    big = torch.full((T, C + 1), float("nan"), dtype=F64, device="cuda")
    big[:, 1:] = Xc
    assert big[:, 1:].data_ptr() % 16 == 8
    out.append(("offset view", big[:, 1:], C + 1))
    return out


def _response(mu, power, rng):
    """A valid response of the family: Poisson counts, compound Poisson-Gamma (exact zeros) for 1 < p < 2, positive
    Gamma draws for p >= 2."""
    if power == 1:
        return rng.poisson(mu).astype(np.float64)
    if power < 2:
        return synth_data.tweedie_draw(mu, int(rng.integers(1 << 30)), power)
    return rng.gamma(2.0, mu / 2.0)


def _row_weights(T, rng, n_w=3):
    """Row-weight vectors with zeros and multiplicities 2 and 3 (eng.index_counts of repeated indices) and a 0/1 fold
    mask; [n_w][ldrw] with ldrw = T + 3."""
    ldrw = T + 3
    RW = torch.zeros((n_w, ldrw), dtype=F64, device="cuda")
    for k in range(n_w):
        if k == 1:
            RW[k, :T] = _dev((rng.random(T) < 0.7).astype(np.float64))
            continue
        idx = rng.integers(0, T, max(T // 2, 1))
        idx = np.concatenate([idx, idx[: max(len(idx) // 3, 1)], idx[:1], idx[:1]])
        RW[k, :T] = eng.index_counts(idx, T)
    return RW, ldrw


# --------------------------------------------------------------------------- reference family terms
def _terms(eta, y, power):
    """Longdouble unit loss l, derivative d = dl/deta, Fisher weight v, each with its magnitude (sum of |parts|)."""
    eta, y = eta.astype(LD), y.astype(LD)
    p = LD(power)
    mu = np.exp(eta)
    mu1 = np.exp((1 - p) * eta)           # mu^(1-p)
    mu2 = np.exp((2 - p) * eta)           # mu^(2-p)
    if power == 1:
        l, lmag = mu - y * eta, mu + np.abs(y * eta)
    elif power == 2:
        l, lmag = eta + y * np.exp(-eta), np.abs(eta) + y * np.exp(-eta)
    else:
        a, b = mu2 / (2 - p), y * mu1 / (1 - p)
        l, lmag = a - b, np.abs(a) + np.abs(b)
    d, dmag = mu1 * (mu - y), mu1 * (mu + y)
    return dict(mu=mu, l=l, lmag=lmag, d=d, dmag=dmag, v=mu2)


def _score_terms(eta, y, power):
    """Longdouble {1, r^2, y, y^2, s4, s5, s6, r} (r = y - mu) and their magnitudes, [8][n]."""
    eta, y = eta.astype(LD), y.astype(LD)
    p = LD(power)
    mu = np.exp(eta)
    one = np.ones_like(eta)
    if power == 1:
        ylogy = np.where(y > 0, y * np.log(np.where(y > 0, y, 1)), 0)
        s, smag = [y * eta, mu, ylogy], [np.abs(y * eta), mu, np.abs(ylogy)]
    elif power == 2:
        s, smag = [eta, y * np.exp(-eta), np.log(y)], [np.abs(eta), y * np.exp(-eta), np.abs(np.log(y))]
    else:
        s = [y * np.exp((1 - p) * eta), np.exp((2 - p) * eta), np.where(y > 0, np.power(y, 2 - p), 0)]
        smag = s
    r = y - mu
    vals = [one, r * r, y, y * y] + s + [r]
    mags = [one, (y + mu) ** 2, y, y * y] + smag + [y + mu]
    return np.stack(vals), np.stack(mags)


def _spread(fn, eta, e):
    """max |fn(eta +- e) - fn(eta)|: the effect of an error e in eta (longdouble)."""
    f0 = fn(eta)
    return np.maximum(np.abs(fn(eta + e) - f0), np.abs(fn(eta - e) - f0))


# --------------------------------------------------------------------------- sglm_pb_eta_f64
def _eta(X, ldx, Wt, ldb, T, C):
    Eta = torch.full((max(T, 1), ldb), float("nan"), dtype=F64, device="cuda")
    eng.call("sglm_pb_eta_f64", eng.ptr(X), ldx, T, C, eng.ptr(Wt), ldb, eng.ptr(Eta), _st())
    return Eta


def _shape_plan(i, T, C):
    ldb = (64, 128, 256)[i % 3]
    B = ldb - 1 if ldb == 64 or (i // 3) % 2 == 0 else 65
    n_live = int(max(4, min(B, MAX_REF_MADDS // max(T * C, 1))))
    return ldb, B, n_live


def _live_columns(B, n_live, rng):
    must = [c for c in (0, 63, 64, 127, 128, B // 2, B - 1) if c < B]
    rest = [c for c in range(B) if c not in must]
    extra = rng.choice(rest, max(0, min(len(rest), n_live - len(must))), replace=False) if rest else []
    return np.array(sorted(set(must) | set(int(c) for c in extra)))


ETA_T = [1, 127, 128, 129, 4097]
ETA_C = [1, 7, 16, 17, 300]


@pytest.mark.parametrize("C", ETA_C)
@pytest.mark.parametrize("T", ETA_T)
def test_pb_eta_matches_longdouble_for_every_layout(T, C):
    i = ETA_T.index(T) * len(ETA_C) + ETA_C.index(C)
    rng = np.random.default_rng(1000 + i)
    ldb, B, n_live = _shape_plan(i, T, C)
    X = _lag_design(T, C, i) if i % 2 == 0 else _wide(T, C, rng)
    live = _live_columns(B, n_live, rng)
    W = np.zeros((C, ldb))
    W[:, live] = rng.standard_normal((C, len(live)))
    W[:, B:] = np.nan                                      # padding columns: never part of a model
    Wt = _dev(W)
    outs = {name: _eta(Xv, ldx, Wt, ldb, T, C) for name, Xv, ldx in _layouts(X)}
    got = outs["ldx=C"][:T, :B].cpu().numpy()
    ref = X.astype(LD) @ W[:, live].astype(LD)
    _check(got[:, live], ref, _sum_bound(C, (np.abs(X) @ np.abs(W[:, live])).astype(LD)), f"eta T={T} C={C} B={B}")
    dead = np.setdiff1d(np.arange(B), live)
    assert np.all(got[:, dead] == 0.0)
    for name, E in outs.items():                           # vector and scalar load paths: the same k order
        _same_bits(E[:T, :B], outs["ldx=C"][:T, :B], f"eta layout {name}")
    W[:, B:] = 0.0
    Xc = _dev(X)
    again = _eta(Xc, C, _dev(W), ldb, T, C)
    _same_bits(again[:T, :B], outs["ldx=C"][:T, :B], "eta with zero instead of NaN padding")


# --------------------------------------------------------------------------- sglm_pb_xt_r_f64
def _xt_r(X, ldx, R, ldb, T, C):
    nbytes = nat.lib().sglm_pb_gemm_tn_workspace_bytes(T, C, ldb)
    ws = torch.full((nbytes // 8 + 2,), float("nan"), dtype=F64, device="cuda")
    Gw = torch.full((C, ldb), float("nan"), dtype=F64, device="cuda")
    eng.call("sglm_pb_xt_r_f64", eng.ptr(X), ldx, T, C, eng.ptr(R), ldb, eng.ptr(Gw), eng.ptr(ws), ws.numel() * 8, _st())
    return Gw


XT_T = [1, 8191, 8192, 8193, 2 * 8192 + 5]
XT_C = [1, 9, 128, 129, 300]


@pytest.mark.parametrize("C", XT_C)
@pytest.mark.parametrize("T", XT_T)
def test_pb_xt_r_matches_longdouble_across_split_boundaries(T, C):
    i = XT_T.index(T) * len(XT_C) + XT_C.index(C)
    rng = np.random.default_rng(2000 + i)
    ldb, B, n_live = _shape_plan(i, T, C)
    X = _lag_design(T, C, i) if i % 2 == 0 else _wide(T, C, rng)
    live = _live_columns(B, n_live, rng)
    R = np.zeros((T, ldb))
    R[:, live] = rng.standard_normal((T, len(live)))
    if T > 2:
        R[rng.random(T) < 0.3, :] = 0.0                    # rows outside a fold
        R[-1, live] = 1.0 + rng.random(len(live))          # the last row of the last split counts
    if T >= 8192:
        R[8191, live] = 3.0                                # last row of the first split, first row of the second
        if T > 8192:
            R[8192, live] = -2.0
    R[:, B:] = np.nan
    Rd = _dev(R)
    outs = {name: _xt_r(Xv, ldx, Rd, ldb, T, C) for name, Xv, ldx in _layouts(X)}
    got = outs["ldx=C"][:, :B].cpu().numpy()
    Rl = R[:, live]
    ref = X.T.astype(LD) @ Rl.astype(LD)
    _check(got[:, live], ref, _sum_bound(T, (np.abs(X).T @ np.abs(Rl)).astype(LD)), f"X'R T={T} C={C} B={B}")
    dead = np.setdiff1d(np.arange(B), live)                # converged models: whole zero columns of R
    assert np.all(got[:, dead] == 0.0)
    for name, G in outs.items():
        _same_bits(G[:, :B], outs["ldx=C"][:, :B], f"X'R layout {name}")
    R[:, B:] = 0.0
    again = _xt_r(_dev(X), C, _dev(R), ldb, T, C)
    _same_bits(again[:, :B], outs["ldx=C"][:, :B], "X'R with zero instead of NaN padding")


# --------------------------------------------------------------------------- sglm_glm_epilogue_f64
class _Batch:
    """Inputs of one epilogue call: Eta [T][ldb] (ldb > n), Y [T][3] (ycol), RW [3][T + 3], b, status."""

    def __init__(self, power, n, T, seed):
        rng = np.random.default_rng(seed)
        self.power, self.n, self.T = power, n, T
        self.ldb = eng._round_up(n + 1, 64)
        self.Eta = np.clip(rng.normal(0.0, 0.8, (max(T, 1), self.ldb)), -2.5, 2.5)
        self.b = rng.uniform(-0.5, 0.5, n)
        self.ldy = 3
        Y = np.stack([_response(np.exp(rng.normal(0.0, 0.5, T)), power, rng) for _ in range(self.ldy)], axis=1)
        if power < 2:
            Y[::7] = 0.0
        self.Y = np.ascontiguousarray(Y)
        self.ycol = np.arange(n, dtype=np.int32) % self.ldy
        self.RWd, self.ldrw = _row_weights(T, rng)
        self.RW = self.RWd.cpu().numpy()[:, :T]
        self.rw_a = np.array([(-1, 0, 1, 2)[k % 4] for k in range(n)], dtype=np.int32)
        self.rw_b = np.array([(-2, -1, 0, 1, 2)[k % 5] for k in range(n)], dtype=np.int32)
        self.status = np.array([(0, 0, 1, 0, 2, 0)[k % 6] for k in range(n)], dtype=np.int32) if n > 1 else \
            np.zeros(1, np.int32)

    def weight(self, rw):
        if rw == -1:
            return np.ones(self.T)
        if rw < -1:
            return np.zeros(self.T)
        return self.RW[rw]

    def run(self, mode, power=None, entry="sglm_glm_epilogue_f64", status=True, Eta=None):
        n, T = self.n, self.T
        Eta = _dev(self.Eta) if Eta is None else Eta
        NS = 4 if mode == 0 else 16
        sums = torch.full((n, NS), float("nan"), dtype=F64, device="cuda")
        nbytes = nat.lib().sglm_pb_epilogue_workspace_bytes(T, n)
        ws = torch.empty(nbytes // 8 + 1, dtype=F64, device="cuda")
        ids = [_dev(a, torch.int32) for a in (self.ycol, self.rw_a, self.rw_b, self.status)]
        Yd, bd = _dev(self.Y), _dev(self.b)
        head = (eng.ptr(Eta), self.ldb, n, T, eng.ptr(Yd), self.ldy, eng.ptr(ids[0]), eng.ptr(self.RWd), self.ldrw,
                eng.ptr(ids[1]), eng.ptr(ids[2]) if mode else None, eng.ptr(bd), eng.ptr(ids[3]) if status else None)
        tail = (mode, eng.ptr(sums), eng.ptr(ws), ws.numel() * 8, _st())
        if entry == "sglm_pb_epilogue_f64":
            eng.call(entry, *head, *tail)
        else:
            eng.call(entry, *head, float(self.power if power is None else power), *tail)
        return Eta, sums


def _epilogue_reference(bt, k):
    """Mode 0 of model k: R [T], sums [4] and their bounds."""
    eta = bt.Eta[:bt.T, k] + bt.b[k]                      # the kernel's own fp64 add: exact input of both sides
    y = bt.Y[:, bt.ycol[k]]
    m = bt.weight(bt.rw_a[k]).astype(LD)
    t = _terms(eta, y, bt.power)
    on = m != 0
    R = np.where(on, m * t["d"], 0)
    Rb = C_ULP * U * np.abs(m) * t["dmag"]
    vals = [m * t["l"], m * t["v"], m, R]
    mags = [np.abs(m) * t["lmag"], np.abs(m) * t["v"], np.abs(m), np.abs(m) * t["dmag"]]
    sums = np.array([np.sum(v) for v in vals])
    bounds = np.array([_sum_bound(bt.T, np.sum(g)) for g in mags])
    return R, Rb, sums, bounds


EPI_SHAPES = [(1, 1), (5, 63), (127, 64), (128, 65), (129, 1), (256, 63), (5, 1184 * 64 + 1), (1, 100003), (129, 4097)]


@pytest.mark.parametrize("n,T", EPI_SHAPES)
@pytest.mark.parametrize("power", POWERS)
def test_glm_epilogue_iteration_mode_matches_longdouble(power, n, T):
    bt = _Batch(power, n, T, seed=hash((power, n, T)) % (1 << 31))
    Eta, sums = bt.run(0)
    got = Eta.cpu().numpy()
    S = sums.cpu().numpy()
    for k in range(n):
        if bt.status[k] != 0:                              # converged / stopped: column untouched, sums zero
            _same_bits(got[:, k], bt.Eta[:, k], f"status {bt.status[k]} model {k} column")
            assert np.all(S[k] == 0.0), (k, S[k])
            continue
        R, Rb, ref, bound = _epilogue_reference(bt, k)
        _check(got[:T, k], R, Rb, f"R p={power} model {k}")
        assert np.all(got[:T, k][bt.weight(bt.rw_a[k]) == 0] == 0.0)
        _check(S[k], ref, bound, f"sums p={power} model {k}")
    _same_bits(got[:, n:], bt.Eta[:, n:], "columns beyond the models")
    Eta2, sums2 = bt.run(0)
    _same_bits(Eta2, Eta, "R of a repeated call")
    _same_bits(sums2, sums, "sums of a repeated call")


@pytest.mark.parametrize("n,T", EPI_SHAPES)
@pytest.mark.parametrize("power", POWERS)
def test_glm_epilogue_score_mode_matches_longdouble(power, n, T):
    bt = _Batch(power, n, T, seed=hash((power, n, T, 1)) % (1 << 31))
    Eta, sums = bt.run(1)
    _same_bits(Eta, bt.Eta, "mode 1 writes no Eta")
    S = sums.cpu().numpy().reshape(n, 2, 8)
    for k in range(n):
        eta = bt.Eta[:T, k] + bt.b[k]
        vals, mags = _score_terms(eta, bt.Y[:, bt.ycol[k]], power)
        for side, rw in ((0, bt.rw_a[k]), (1, bt.rw_b[k])):
            m = bt.weight(rw).astype(LD)
            ref = (vals * m).sum(axis=1)
            bound = _sum_bound(T, (mags * np.abs(m)).sum(axis=1))
            _check(S[k, side], ref, bound, f"score sums p={power} model {k} side {side} rw {rw}")
    _, again = bt.run(1)
    _same_bits(again, sums, "score sums of a repeated call")


def _d2_bound(s, b, power):
    """Bound on D^2 from sums s[0..7] with bounds b[0..7]: each sum's bound and the host's rounding (C_ULP u |s_i|)
    carried linearly through dev and dev_null (tweedie_d2_from_sums)."""
    n, sy = s[0], s[2]
    ybar = sy / n
    if power == 1:
        a_dev = {6: 1.0, 4: 1.0, 2: 1.0, 5: 1.0}
        a_null = {6: 1.0, 2: abs(np.log(ybar)) + 1.0}
    elif power == 2:
        a_dev = {4: 1.0, 6: 1.0, 5: 1.0, 0: 1.0}
        a_null = {6: 1.0, 2: 1.0 / ybar, 0: abs(np.log(ybar)) + 1.0}
    else:
        p = power
        a_dev = {6: 1 / abs((1 - p) * (2 - p)), 4: 1 / abs(1 - p), 5: 1 / abs(2 - p)}
        a_null = {6: 1 / abs((1 - p) * (2 - p)), 2: ybar ** (1 - p) / abs(1 - p), 0: ybar ** (2 - p) / abs(2 - p)}
    e = lambda a: 2.0 * sum(c * (b[i] + C_ULP * U * abs(s[i])) for i, c in a.items())
    return eng.tweedie_d2_from_sums(s, power), e(a_dev), e(a_null)


def _unit_deviance(y, mu, power):
    y, mu = y.astype(LD), mu.astype(LD)
    p = LD(power)
    if power == 1:
        return 2 * (np.where(y > 0, y * np.log(np.where(y > 0, y, 1) / mu), 0) - y + mu)
    if power == 2:
        return 2 * (np.log(mu / y) + y / mu - 1)
    return 2 * (np.power(y, 2 - p) / ((1 - p) * (2 - p)) - y * np.power(mu, 1 - p) / (1 - p)
                + np.power(mu, 2 - p) / (2 - p))


@pytest.mark.parametrize("case", ["gamma_low_dispersion", "poisson_counts_1e3", "tweedie_1.5"])
def test_d2_from_kernel_sums_matches_unit_deviances(case):
    """D^2 from the mode-1 sums against D^2 from per-row unit deviances.  Low-dispersion Gamma and Poisson counts near
    1e3 are where the sums-based deviance cancels most: dev is a small difference of large sums."""
    T, n = 100003, 4
    rng = np.random.default_rng(11)
    power = {"gamma_low_dispersion": 2.0, "poisson_counts_1e3": 1.0, "tweedie_1.5": 1.5}[case]
    bt = _Batch(power, n, T, seed=12)
    base = {2.0: 0.0, 1.0: np.log(1000.0), 1.5: 0.0}[power]
    bt.b = np.full(n, base) + rng.uniform(-0.1, 0.1, n)
    z = rng.normal(0.0, 0.3, T)
    for k in range(n):
        bt.Eta[:T, k] = z + rng.normal(0.0, 0.01, T)
    mu_true = np.exp(z + base)
    if power == 2:
        y = mu_true * rng.gamma(1e4, 1e-4, T)              # dispersion 1e-4
    elif power == 1:
        y = rng.poisson(mu_true).astype(np.float64)
    else:
        y = synth_data.tweedie_draw(mu_true, 3, 1.5)
    bt.Y = np.ascontiguousarray(np.repeat(y[:, None], 3, axis=1))
    bt.rw_a = np.array([-1, 0, 1, 2], dtype=np.int32)
    bt.rw_b = np.array([1, -1, 2, 0], dtype=np.int32)
    _, sums = bt.run(1)
    S = sums.cpu().numpy().reshape(n, 2, 8)
    worst = 0.0
    for k in range(n):
        eta = bt.Eta[:T, k] + bt.b[k]
        vals, mags = _score_terms(eta, y, power)
        mu = np.exp(eta.astype(LD))
        for side, rw in ((0, bt.rw_a[k]), (1, bt.rw_b[k])):
            m = bt.weight(rw).astype(LD)
            ybar = np.sum(m * y) / np.sum(m)
            dev = np.sum(m * _unit_deviance(y, mu, power))
            dev_null = np.sum(m * _unit_deviance(y, np.full(T, ybar, dtype=LD), power))
            ref = 1 - dev / dev_null
            sb = _sum_bound(T, (mags * np.abs(m)).sum(axis=1)).astype(np.float64)
            d2, e_dev, e_null = _d2_bound(S[k, side], sb, power)
            bound = (e_dev + abs(1 - d2) * e_null) / float(dev_null)
            err = abs(LD(d2) - ref)
            worst = max(worst, float(err))
            assert err <= bound, (case, k, side, d2, float(ref), float(err), bound)
    print(f"\nD2 {case}: largest |D2(kernel sums) - D2(longdouble unit deviances)| = {worst:.3e}")


# --------------------------------------------------------------------------- invariants across entry points / positions
@pytest.mark.parametrize("power", [1.0, 1.5])
def test_model_outputs_do_not_depend_on_position_or_neighbours(power):
    T, C = 4097 + 8192, 33
    rng = np.random.default_rng(5)
    X = _lag_design(T, C, 5)
    Xd = _dev(X)
    w = rng.normal(0.0, 0.2, C)
    y = _response(np.exp(rng.normal(0, 0.5, T)), power, rng)
    RWd, ldrw = _row_weights(T, rng)
    b = -0.3

    def chain(ldb, n, pos):
        W = rng.normal(0.0, 0.2, (C, ldb))
        W[:, n:] = np.nan
        W[:, pos] = w
        Eta = _eta(Xd, C, _dev(W), ldb, T, C)
        Y = np.ascontiguousarray(rng.gamma(2.0, 1.0, (T, 2)))
        Y[:, 1] = y
        ycol = rng.integers(0, 2, n).astype(np.int32)
        rw_a = rng.integers(-1, 3, n).astype(np.int32)
        rw_b = rng.integers(-2, 3, n).astype(np.int32)
        bv = rng.uniform(-1, 1, n)
        ycol[pos], rw_a[pos], rw_b[pos], bv[pos] = 1, 0, 2, b
        st = np.zeros(n, np.int32)
        ids = [_dev(a, torch.int32) for a in (ycol, rw_a, rw_b, st)]
        Yd, bd = _dev(Y), _dev(bv)
        out = [Eta[:, pos].clone()]
        for mode in (1, 0):
            sums = torch.empty((n, 16 if mode else 4), dtype=F64, device="cuda")
            ws = torch.empty(nat.lib().sglm_pb_epilogue_workspace_bytes(T, n) // 8 + 1, dtype=F64, device="cuda")
            eng.call("sglm_glm_epilogue_f64", eng.ptr(Eta), ldb, n, T, eng.ptr(Yd), 2, eng.ptr(ids[0]), eng.ptr(RWd),
                     ldrw, eng.ptr(ids[1]), eng.ptr(ids[2]), eng.ptr(bd), eng.ptr(ids[3]), power, mode, eng.ptr(sums),
                     eng.ptr(ws), ws.numel() * 8, _st())
            out.append(sums[pos].clone())
        out.append(Eta[:, pos].clone())
        Eta[:, n:] = float("nan")
        out.append(_xt_r(Xd, C, Eta, ldb, T, C)[:, pos].clone())
        return out

    alone = chain(64, 1, 0)
    for pos in (127, 128, 129, 255):
        got = chain(256, 256, pos)
        for what, a, g in zip(("eta", "score sums", "sums", "R", "X'R"), alone, got):
            _same_bits(g, a, f"{what} at position {pos}")


def test_poisson_entry_points_equal_the_family_ones_at_power_1():
    T, C = 3001, 21
    rng = np.random.default_rng(9)
    bt = _Batch(1.0, 40, T, seed=9)
    for mode in (0, 1):
        Ea, sa = bt.run(mode, entry="sglm_pb_epilogue_f64")
        Eb, sb = bt.run(mode, power=1.0)
        _same_bits(Ea, Eb, f"pb vs glm epilogue R, mode {mode}")
        _same_bits(sa, sb, f"pb vs glm epilogue sums, mode {mode}")
    X = _dev(_lag_design(T, C, 9))
    y = _dev(rng.poisson(1.5, T).astype(np.float64))
    rw = eng.index_counts(np.concatenate([np.arange(0, T, 2), np.arange(0, T, 5)]), T)
    w, b = _dev(rng.normal(0, 0.1, C)), _dev([0.2])
    ws = torch.empty(nat.lib().sglm_score_workspace_bytes() // 8, dtype=F64, device="cuda")
    outs = []
    for entry in ("sglm_score_f64", "sglm_score_glm_f64"):
        r, s = torch.empty(T, dtype=F64, device="cuda"), torch.empty(8, dtype=F64, device="cuda")
        mid = 1 if entry == "sglm_score_f64" else 1.0
        eng.call(entry, eng.ptr(X), C, eng.ptr(y), eng.ptr(rw), T, C, eng.ptr(w), eng.ptr(b), mid, eng.ptr(r),
                 eng.ptr(s), eng.ptr(ws), _st())
        outs.append((r, s))
    _same_bits(outs[0][0], outs[1][0], "score residuals")
    _same_bits(outs[0][1], outs[1][1], "score sums")
    outs = []
    for entry in ("sglm_poisson_irls_prepare_f64", "sglm_glm_irls_prepare_f64"):
        o0, o1 = torch.empty(T, dtype=F64, device="cuda"), torch.empty(T, dtype=F64, device="cuda")
        s = torch.empty(8, dtype=F64, device="cuda")
        extra = () if entry == "sglm_poisson_irls_prepare_f64" else (1.0,)
        eng.call(entry, eng.ptr(X), C, eng.ptr(y), eng.ptr(rw), T, C, eng.ptr(w), eng.ptr(b), *extra, eng.ptr(o0),
                 eng.ptr(o1), eng.ptr(s), eng.ptr(ws), _st())
        outs.append((o0, o1, s[:4]))
    for what, a, g in zip(("weight", "working response", "sums"), outs[0], outs[1]):
        _same_bits(a, g, f"irls prepare {what}")


# --------------------------------------------------------------------------- row passes (predict.cu)
ROW_CASES = [(5, 7, "ldx=C"), (300, 33, "ldx=C+1"), (300, 32, "ldx=C+1"), (1000, 17, "offset view"),
             (2000, 32, "offset view"), ("big", 9, "ldx=C"), (16, 25600, "ldx=C")]


@pytest.mark.parametrize("T,C,layout", ROW_CASES)
@pytest.mark.parametrize("power", [1.0, 2.0, 1.5, 3.0])
def test_row_passes_match_longdouble(power, T, C, layout):
    if T == "big":
        T = 8 * _sms() * 8 + 1000           # grid-stride loop, more than 256 partials in finish_sums_kernel
    rng = np.random.default_rng(C * 7 + T)
    X = _lag_design(T, C, C)
    Xv, ldx = {name: (v, l) for name, v, l in _layouts(X)}[layout]
    w = rng.normal(0.0, 0.3 / np.sqrt(C), C)
    b = -0.2
    wd, bd = _dev(w), _dev([b])
    y = _response(np.exp(rng.normal(0.0, 0.5, T)), power, rng)
    if power < 2:
        y[::5] = 0.0
    RWd, _ = _row_weights(T, rng, 1)
    rw = RWd[0, :T].contiguous()
    m = rw.cpu().numpy().astype(LD)
    yd = _dev(y)
    eta_ref = X.astype(LD) @ w.astype(LD) + LD(b)
    e = _sum_bound(C + 1, (np.abs(X) @ np.abs(w) + abs(b)).astype(LD))
    assert np.max(np.abs(eta_ref)) < 3.0
    # predict, identity and log link
    for link in (0, 1):
        out = torch.full((T,), float("nan"), dtype=F64, device="cuda")
        eng.call("sglm_predict_f64", eng.ptr(Xv), ldx, T, C, eng.ptr(wd), eng.ptr(bd), link, eng.ptr(out), _st())
        if link == 0:
            _check(out.cpu().numpy(), eta_ref, e, f"predict link 0 {layout}")
        else:
            _check(out.cpu().numpy(), np.exp(eta_ref), _spread(np.exp, eta_ref, e) + C_ULP * U * np.exp(eta_ref),
                   f"predict link 1 {layout}")
    ws = torch.empty(nat.lib().sglm_score_workspace_bytes() // 8, dtype=F64, device="cuda")
    # score: residuals and 8 sums
    r = torch.full((T,), float("nan"), dtype=F64, device="cuda")
    s = torch.full((8,), float("nan"), dtype=F64, device="cuda")
    eng.call("sglm_score_glm_f64", eng.ptr(Xv), ldx, eng.ptr(yd), eng.ptr(rw), T, C, eng.ptr(wd), eng.ptr(bd), power,
             eng.ptr(r), eng.ptr(s), eng.ptr(ws), _st())
    mu_ref = np.exp(eta_ref)
    _check(r.cpu().numpy(), y - mu_ref, _spread(np.exp, eta_ref, e) + C_ULP * U * (y + mu_ref), "score residual")
    vals, mags = _score_terms(eta_ref, y, power)
    spread = np.stack([_spread(lambda t, i=i: _score_terms(t, y, power)[0][i], eta_ref, e) for i in range(8)])
    ref = (vals * m).sum(axis=1)
    bound = _sum_bound(T, (mags * np.abs(m)).sum(axis=1)) + (spread * np.abs(m)).sum(axis=1)
    _check(s.cpu().numpy(), ref, bound, f"score sums p={power}")
    # IRLS preparation: Fisher weight, working response, 4 sums
    o0 = torch.full((T,), float("nan"), dtype=F64, device="cuda")
    o1 = torch.full((T,), float("nan"), dtype=F64, device="cuda")
    s = torch.full((8,), float("nan"), dtype=F64, device="cuda")
    eng.call("sglm_glm_irls_prepare_f64", eng.ptr(Xv), ldx, eng.ptr(yd), eng.ptr(rw), T, C, eng.ptr(wd), eng.ptr(bd),
             power, eng.ptr(o0), eng.ptr(o1), eng.ptr(s), eng.ptr(ws), _st())
    on = m != 0
    t = _terms(eta_ref, y, power)
    v_spread = _spread(lambda q: _terms(q, y, power)["v"], eta_ref, e)
    z = eta_ref + (y - t["mu"]) / t["mu"]
    z_fn = lambda q: q + (y - np.exp(q)) / np.exp(q)
    z_bound = _spread(z_fn, eta_ref, e) + C_ULP * U * (np.abs(eta_ref) + y / t["mu"] + 1)
    got0, got1 = o0.cpu().numpy(), o1.cpu().numpy()
    _check(got0, np.where(on, m * t["v"], 0), np.abs(m) * (v_spread + C_ULP * U * t["v"]), f"Fisher weight p={power}")
    _check(got1, np.where(on, z, 0), np.where(on, z_bound, 0), f"working response p={power}")
    assert np.all(got0[~on] == 0.0) and np.all(got1[~on] == 0.0)
    l_spread = _spread(lambda q: _terms(q, y, power)["l"], eta_ref, e)
    ref = np.array([np.sum(m * t["l"]), np.sum(m * t["v"]), np.sum(m), np.sum(m * y)])
    bound = np.array([_sum_bound(T, np.sum(np.abs(m) * t["lmag"])) + np.sum(np.abs(m) * l_spread),
                      _sum_bound(T, np.sum(np.abs(m) * t["v"])) + np.sum(np.abs(m) * v_spread),
                      _sum_bound(T, np.sum(np.abs(m))), _sum_bound(T, np.sum(np.abs(m) * y))])
    _check(s[:4].cpu().numpy(), ref, bound, f"irls sums p={power}")


@pytest.mark.parametrize("T,C,layout", [(2000, 1023, "ldx=C"), (2000, 1024, "ldx=C+1"), (2000, 1025, "offset view"),
                                        (900, 2100, "ldx=C+3"), (5, 3, "ldx=C"), (70001, 5, "ldx=C+1")])
def test_xt_vec_matches_longdouble(T, C, layout):
    rng = np.random.default_rng(T + C)
    X = _wide(T, C, rng) if C % 2 else _lag_design(T, C, 3)
    Xv, ldx = {name: (v, l) for name, v, l in _layouts(X)}[layout]
    r = rng.standard_normal(T)
    r[rng.random(T) < 0.3] = 0.0                              # rows outside the fold
    nbytes = nat.lib().sglm_xt_vec_workspace_bytes(C)
    ws = torch.full((nbytes // 8,), float("nan"), dtype=F64, device="cuda")
    out = torch.full((C,), float("nan"), dtype=F64, device="cuda")
    rd = _dev(r)
    eng.call("sglm_xt_vec_f64", eng.ptr(Xv), ldx, eng.ptr(rd), T, C, eng.ptr(out), eng.ptr(ws), nbytes, _st())
    ref = X.T.astype(LD) @ r.astype(LD)
    _check(out.cpu().numpy(), ref, _sum_bound(T, (np.abs(X).T @ np.abs(r)).astype(LD)), f"X'r T={T} C={C} {layout}")
    again = torch.full((C,), float("nan"), dtype=F64, device="cuda")
    eng.call("sglm_xt_vec_f64", eng.ptr(Xv), ldx, eng.ptr(rd), T, C, eng.ptr(again), eng.ptr(ws), nbytes, _st())
    _same_bits(again, out, "X'r of a repeated call")


# --------------------------------------------------------------------------- empty row slice (T = 0)
def test_empty_row_slice_writes_zero_sums_with_null_row_pointers():
    """An empty torch tensor's data_ptr() is 0: a rank of a row-sharded batch that holds no rows passes NULL."""
    C, n, ldb = 7, 5, 64
    nan = float("nan")
    w, b = _dev(np.ones(C)), _dev([0.5])
    ws = torch.empty(nat.lib().sglm_score_workspace_bytes() // 8, dtype=F64, device="cuda")
    for power in (1.0, 2.0, 1.5):
        s = torch.full((8,), nan, dtype=F64, device="cuda")
        eng.call("sglm_score_glm_f64", None, C, None, None, 0, C, eng.ptr(w), eng.ptr(b), power, None, eng.ptr(s),
                 eng.ptr(ws), _st())
        assert torch.all(s == 0), s
        s = torch.full((8,), nan, dtype=F64, device="cuda")
        eng.call("sglm_glm_irls_prepare_f64", None, C, None, None, 0, C, eng.ptr(w), eng.ptr(b), power, None, None,
                 eng.ptr(s), eng.ptr(ws), _st())
        assert torch.all(s[:4] == 0), s
        ids = _dev(np.array([0, 1, 0, 1, 0]), torch.int32)
        rw_a = _dev(np.array([-1, 0, 1, -1, 2]), torch.int32)       # ids >= 0 name rows of an empty RW
        rw_b = _dev(np.array([-2, -1, 0, 1, 2]), torch.int32)
        st = _dev(np.zeros(n), torch.int32)
        bv = _dev(np.zeros(n))
        for mode in (0, 1):
            sums = torch.full((n, 16 if mode else 4), nan, dtype=F64, device="cuda")
            nb = nat.lib().sglm_pb_epilogue_workspace_bytes(0, n)
            ews = torch.empty(nb // 8 + 1, dtype=F64, device="cuda")
            eng.call("sglm_glm_epilogue_f64", None, ldb, n, 0, None, 2, eng.ptr(ids), None, 0, eng.ptr(rw_a),
                     eng.ptr(rw_b) if mode else None, eng.ptr(bv), eng.ptr(st), power, mode, eng.ptr(sums), eng.ptr(ews),
                     ews.numel() * 8, _st())
            assert torch.all(sums == 0), (power, mode, sums)
    nb = nat.lib().sglm_pb_gemm_tn_workspace_bytes(0, C, ldb)
    xws = torch.empty(nb // 8 + 2, dtype=F64, device="cuda")
    Gw = torch.full((C, ldb), nan, dtype=F64, device="cuda")
    eng.call("sglm_pb_xt_r_f64", None, C, 0, C, None, ldb, eng.ptr(Gw), eng.ptr(xws), xws.numel() * 8, _st())
    assert torch.all(Gw == 0)
    nb = nat.lib().sglm_xt_vec_workspace_bytes(C)
    vws = torch.empty(nb // 8, dtype=F64, device="cuda")
    out = torch.full((C,), nan, dtype=F64, device="cuda")
    eng.call("sglm_xt_vec_f64", None, C, None, 0, C, eng.ptr(out), eng.ptr(vws), nb, _st())
    assert torch.all(out == 0)
    eng.call("sglm_pb_eta_f64", None, C, 0, C, None, ldb, None, _st())


# --------------------------------------------------------------------------- sglm_pb_step_f64
# Models of the step test, one per branch:
#   0 already done (status 1)            1 worse objective, halv < 30: halving      2 worse, halv = 30: a step
#   3 n_iter = max_iter: status 2        4 first step after a refresh (no previous step known)
#   5 no intercept, last step >= 1e300   6 hscale != 1, meets the rho rule           7 fails the rho rule
STEP_B = 8


def _step_setup(C, rng):
    B, ldw, ldq, ldb = STEP_B, eng._round_up(C, 2), eng._round_up(C, 8), 64
    Q, xbar, h11 = [], [], []
    for _ in range(2):
        A = rng.standard_normal((C, C))
        Q.append(A @ A.T / C + 0.5 * np.eye(C))
        xbar.append(rng.uniform(-0.3, 0.3, C))
        h11.append(rng.uniform(50.0, 200.0))
    s = dict(C=C, B=B, ldw=ldw, ldq=ldq, ldb=ldb, Q=Q, xbar=xbar, h11=np.array(h11))
    s["hess_id"] = np.array([0, 1, 0, 1, 0, 1, 0, 1], np.int32)
    s["fit_icpt"] = np.array([1, 1, 1, 1, 1, 0, 1, 1], np.int32)
    s["alpha"] = rng.uniform(1e-3, 1e-1, B)
    s["n_tot"] = rng.uniform(100.0, 1000.0, B)
    s["hscale"] = np.array([1, 1, 2.5, 1, 1, 1, 0.37, 1.0])
    s["an"] = s["alpha"] * s["n_tot"] / s["hscale"] * np.array([1, 1, 1.1, 1, 1, 1, 0.8, 1])   # the factors' shifts
    s["tol"] = np.full(B, 1e-4)
    s["max_iter"] = np.array([100, 100, 100, 7, 100, 100, 100, 100], np.int32)
    s["n_iter"] = np.array([3, 4, 5, 7, 0, 2, 6, 6], np.int32)
    s["status"] = np.array([1, 0, 0, 0, 0, 0, 0, 0], np.int32)
    s["halv"] = np.array([0, 3, 30, 0, 0, 0, 0, 0], np.int32)
    s["has_prev"] = np.array([1, 1, 1, 1, 0, 1, 1, 1], np.int32)
    W = np.zeros((B, ldw))
    W[:, :C] = rng.uniform(-0.9, 0.9, (B, C))
    Wp = np.zeros((B, ldw))
    Wp[:, :C] = rng.uniform(-0.9, 0.9, (B, C))
    s["W"], s["Wprev"] = W, Wp
    s["b"], s["bprev"] = rng.uniform(-1, 1, B), rng.uniform(-1, 1, B)
    sums = np.zeros((B, 4))
    sums[:, 0] = rng.uniform(50.0, 500.0, B)
    sums[:, 3] = rng.normal(0.0, 2.0, B)
    sums[[6, 7], 3] = 0.0
    s["sums"] = sums
    f = sums[:, 0] / s["n_tot"] + 0.5 * s["alpha"] * np.sum(W[:, :C] ** 2, axis=1)
    worse = np.array([0, 1, 1, 0, 0, 0, 0, 0], bool)
    s["fprev"] = np.where(worse, f - 1.0, f + 1.0)
    Gw = np.zeros((C, ldb))
    Gw[:, :B] = rng.normal(0.0, 1.0, (C, B))
    delta = 4e-9                                            # models 6 and 7: w_new = w + delta e_0
    for k in (6, 7):
        A = Q[s["hess_id"][k]].astype(LD) + LD(s["an"][k]) * np.eye(C, dtype=LD)
        w = W[k, :C].astype(LD)
        wt = w.copy()
        wt[0] += LD(delta)
        need = A @ wt - Q[s["hess_id"][k]].astype(LD) @ w
        Gw[:, k] = np.asarray(-LD(s["hscale"][k]) * need, dtype=np.float64)
    s["Gw"] = Gw
    s["last_step"] = np.array([0.5, 0.5, 0.3, 0.5, 0.0, 2e300, 10 * delta, 10 * delta])
    s["ratio_out"] = np.array([0.7, 0.7, 0.4, 0.7, 1.0, 0.6, 0.5, 0.9])
    return s


def _step_run(s):
    C, B, ldw, ldq = s["C"], s["B"], s["ldw"], s["ldq"]
    d = {}
    for k in ("W", "Wprev", "b", "bprev", "fprev", "last_step", "ratio_out", "alpha", "n_tot", "tol", "sums", "Gw",
              "hscale"):
        d[k] = _dev(s[k])
    d["Wnew"] = torch.full((B, ldw), float("nan"), dtype=F64, device="cuda")
    d["rhs"] = torch.zeros((B, ldw), dtype=F64, device="cuda")
    d["fcur"] = torch.full((B,), -7.0, dtype=F64, device="cuda")
    d["step_out"] = torch.full((B,), -7.0, dtype=F64, device="cuda")
    for k in ("halv", "n_iter", "status", "has_prev", "fit_icpt", "max_iter", "hess_id"):
        d[k] = _dev(s[k], torch.int32)
    d["flag"] = torch.full((B,), -7, dtype=torch.int32, device="cuda")
    Qd, xb = [], []
    for g in range(2):
        q = torch.zeros((C, ldq), dtype=F64, device="cuda")
        q[:, :C] = _dev(s["Q"][g])
        Qd.append(q)
        xb.append(_dev(s["xbar"][g]))
    d["HQ"] = _dev(np.array([q.data_ptr() for q in Qd], np.int64), torch.int64)
    d["Hxbar"] = _dev(np.array([x.data_ptr() for x in xb], np.int64), torch.int64)
    d["Hh11"] = _dev(s["h11"])
    # the factors of (Q_g + an_k I), as _poisson_batch's refresh() makes them
    L_of = np.zeros(B, np.int64)
    keep = [Qd, xb]
    for g in range(2):
        idx = np.flatnonzero(s["hess_id"] == g)
        an = _dev(s["an"][idx])
        wb = nat.lib().sglm_ridge_workspace_bytes(C, ldq, len(idx))
        work = torch.empty(wb // 8, dtype=F64, device="cuda")
        Wtmp = torch.empty((len(idx), ldw), dtype=F64, device="cuda")
        st = torch.empty(len(idx), dtype=torch.int32, device="cuda")
        qc = torch.zeros(C, dtype=F64, device="cuda")
        eng.call("sglm_ridge_solve_f64", eng.ptr(Qd[g]), ldq, eng.ptr(qc), C, eng.ptr(an), len(idx), eng.ptr(Wtmp), ldw,
                 eng.ptr(st), eng.ptr(work), wb, _st())
        assert torch.all(st == 0)
        for j, k in enumerate(idx):
            L_of[k] = work.data_ptr() + j * (C + 1) * ldq * 8
        keep += [an, work, Wtmp, st, qc]
    L_of_d = _dev(L_of, torch.int64)
    order = ["W", "Wprev", "Wnew", "rhs", "b", "bprev", "fprev", "fcur", "last_step", "step_out", "ratio_out", "halv",
             "n_iter", "status", "flag", "has_prev", "alpha", "n_tot", "tol", "fit_icpt", "max_iter", "hess_id", "HQ",
             "Hxbar", "Hh11", "sums", "Gw", "hscale"]
    words = [d[k].data_ptr() for k in order] + [ldw, ldq, s["ldb"], C | (B << 32)]
    assert len(words) == nat.lib().sglm_pb_state_words()
    state = np.array(words, dtype=np.uint64)
    eng.call("sglm_pb_step_f64", state.ctypes.data_as(ctypes.c_void_p), eng.ptr(L_of_d), _st())
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in d.items()}


@pytest.mark.parametrize("C", [5, 33, 300])
def test_pb_step_visits_every_branch_as_documented(C):
    rng = np.random.default_rng(C)
    s = _step_setup(C, rng)
    o = _step_run(s)
    again = _step_run(s)
    for k in o:
        if k not in ("HQ", "Hxbar"):                           # device pointers of each run's own buffers
            _same_bits(again[k], o[k], f"repeated step: {k}")
    B, W0 = s["B"], s["W"]
    expect_flag = np.array([0, 2, 1, 0, 1, 1, 1, 1])
    assert np.array_equal(o["flag"], expect_flag), o["flag"]
    for k in range(B):
        w0 = W0[k, :C]
        hid, icpt, hs = s["hess_id"][k], bool(s["fit_icpt"][k]), s["hscale"][k]
        f_ref = LD(s["sums"][k, 0]) / LD(s["n_tot"][k]) + LD(0.5) * LD(s["alpha"][k]) * np.sum(w0.astype(LD) ** 2)
        if expect_flag[k] == 0:                                # done / stopped: nothing moves but status
            assert o["step_out"][k] == 0.0
            for key in ("W", "Wprev", "b", "bprev", "fprev", "last_step", "ratio_out", "n_iter", "halv", "has_prev"):
                _same_bits(o[key][k], s[key][k], f"model {k} {key}")
            assert o["status"][k] == (1 if k == 0 else 2)
            continue
        if expect_flag[k] == 2:                                # halving towards the previous iterate
            assert o["step_out"][k] == -1.0 and o["halv"][k] == s["halv"][k] + 1 and o["status"][k] == 0
            _same_bits(o["W"][k], 0.5 * (W0[k] + s["Wprev"][k]), "halved w")
            _same_bits(o["b"][k], 0.5 * (s["b"][k] + s["bprev"][k]), "halved b")
            for key in ("Wprev", "bprev", "fprev", "last_step", "ratio_out", "n_iter", "has_prev"):
                _same_bits(o[key][k], s[key][k], f"model {k} {key}")
            continue
        # a chord step: rhs = Q w + (-g + xbar g_b) / hs, (Q + an I) w_new = rhs
        Q = s["Q"][hid].astype(LD)
        xbar = s["xbar"][hid]
        g_b = s["sums"][k, 3]
        extra = (-s["Gw"][:C, k].astype(LD) + (xbar.astype(LD) * LD(g_b) if icpt else 0)) / LD(hs)
        rhs_ref = Q @ w0.astype(LD) + extra
        rhs_mag = np.abs(s["Q"][hid]) @ np.abs(w0) + (np.abs(s["Gw"][:C, k]) + (np.abs(xbar * g_b) if icpt else 0)) / hs
        _check(o["rhs"][k, :C], rhs_ref, _sum_bound(C + 2, rhs_mag.astype(LD)), f"rhs model {k}")
        A = s["Q"][hid] + s["an"][k] * np.eye(C)
        w_ref = np.linalg.solve(A.astype(np.float64), np.asarray(rhs_ref, dtype=np.float64)).astype(LD)
        for _ in range(2):                                     # refine in longdouble
            w_ref = w_ref + np.linalg.solve(A, np.asarray(rhs_ref - A.astype(LD) @ w_ref, dtype=np.float64)).astype(LD)
        sv = np.linalg.svd(A, compute_uv=False)
        kappa, inv_norm = sv[0] / sv[-1], 1.0 / sv[-1]
        w_bound = C_ULP * C * U * (kappa * np.linalg.norm(np.asarray(w_ref, dtype=np.float64)) +
                                   inv_norm * np.linalg.norm(rhs_mag))
        wn = o["Wnew"][k, :C]
        err = float(np.linalg.norm(np.asarray(wn.astype(LD) - w_ref, dtype=np.float64)))
        assert err <= w_bound, (k, err, w_bound)
        _same_bits(o["W"][k, :C], wn, "w <- w_new")
        _same_bits(o["Wprev"][k], W0[k], "w_prev <- w")
        # intercept, step, convergence: the documented step on the kernel's w_new
        dw = wn - w0
        b_old = s["b"][k]
        if icpt:
            b_ref = LD(b_old) - LD(g_b) / (LD(s["h11"][hid]) * LD(hs)) - np.sum(xbar.astype(LD) * dw.astype(LD))
            b_mag = abs(b_old) + abs(g_b / (s["h11"][hid] * hs)) + np.sum(np.abs(xbar * dw))
            _check(np.array([o["b"][k]]), np.array([b_ref]), np.array([_sum_bound(C + 3, LD(b_mag))]), f"b model {k}")
        else:
            assert o["b"][k] == 0.0
        b_new = o["b"][k]
        step = max(np.max(np.abs(dw)), abs(b_new - b_old)) / max(1.0, np.max(np.abs(wn)))
        last = s["last_step"][k]
        have = 0.0 < last < 1e300
        ratio = step / last if have else 1.0
        rho = min(max(ratio, s["ratio_out"][k]), 0.9)
        done = step * rho / (1.0 - rho) <= min(s["tol"][k], 1e-8) or step <= 1e-12
        assert o["step_out"][k] == step and o["last_step"][k] == step and o["ratio_out"][k] == ratio, k
        assert o["status"][k] == (1 if done else 0), (k, step, rho)
        assert o["n_iter"][k] == s["n_iter"][k] + 1 and o["halv"][k] == 0 and o["has_prev"][k] == 1
        _same_bits(o["bprev"][k], b_old, "b_prev <- b")
        _check(o["fcur"][k:k + 1], np.array([f_ref]),
               np.array([_sum_bound(C + 2, LD(s["sums"][k, 0] / s["n_tot"][k]) + LD(0.5 * s["alpha"][k]) *
                                    np.sum(w0.astype(LD) ** 2))]), f"objective model {k}")
        _same_bits(o["fprev"][k], o["fcur"][k], "f_prev <- f")
    # the designed outcomes: model 6 converges by the rho rule, model 7 (the worse of the last two ratios is 0.9)
    # does not although its own ratio is 0.1; the first step after a refresh cannot converge
    assert o["status"][6] == 1 and o["status"][7] == 0 and o["status"][4] == 0
    assert 0.05 < o["ratio_out"][7] < 0.2 and o["ratio_out"][4] == 1.0 and o["ratio_out"][5] == 1.0
